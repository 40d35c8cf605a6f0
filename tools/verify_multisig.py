#!/usr/bin/env python
"""Measures blsgpu_verify_multisig_batch[_keyed] and blsgpu_sum_points_batch against what a caller had to do before them
(one blsgpu_sum_points call per multi-signature, then one blsgpu_verify_batch call), and against keyed verify_secure on the
same quorums.

Shapes (a multi-signature of set j is [sum of its signers' secrets] H(msg_j), from blsgpu_testdata_sign; 32-byte messages):
  A    10,000 multi-signatures x 400 distinct signers drawn from a 2^16-key set, Bls12381G2Impl, ProofOfPossession, Modern:
       keyed vs unkeyed vs the loop (blsgpu_sum_points timed over the first 100 sets and reported per set, then one
       blsgpu_verify_batch on the q sums), and blsgpu_verify_secure_batch_keyed on the same quorums (its own aggregates)
  A1   A for Bls12381G1Impl: keyed vs unkeyed
  B    one multi-signature of 2^20 signers (a 2^20-key set): keyed vs blsgpu_sum_points of the keys + blsgpu_verify_batch
  C    2^18 sets x 2 signers: keyed vs blsgpu_verify_batch on the pre-summed keys
  D    A with 1 and with 100 wrong multi-signatures (signatures of another set) against A
  E    blsgpu_sum_points_batch over 10,000 x 400 signatures vs blsgpu_sum_points per set (the first 100 sets, per set)
Calls alternate after a warm-up of each; wall clock around each call (every call ends in a stream synchronisation), and
blsgpu_last_stage_ms of the keyed calls (the key sums are the decode_pk stage).  Every status vector (and sum) must match
across the calls compared, or the tool stops.  The sum stage's share of the IMAD peak: M mixed additions x (11 Fp-mul in G1,
29 in G2) x 300 MACs over the stage's device time over blsgpu_imad_peak.

    python tools/verify_multisig.py --out DIR [--reps 3]   -> DIR/verify_multisig_b200.json
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "agora-blsful_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)
sys.dont_write_bytecode = True

import numpy as np

R = 0x73EDA753299D7D483339D80809A1D80553BDA402FFFE5BFEFFFFFFFF00000001
MEM, Q, KEYS = 400, 10_000, 1 << 16
FP_MUL = {1: 11, 2: 29}   # Fp multiplications per mixed addition in G1 / G2 (SURVEY section 8d), 300 MACs each


def device_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"unavailable: {e}"


def timed(f):
    t = time.perf_counter()
    r = f()
    return r, (time.perf_counter() - t) * 1e3


def secrets(rng, n):
    s = np.zeros((n, 32), dtype=np.uint8)
    s[:, 8:] = rng.integers(0, 256, size=(n, 24), dtype=np.uint8)
    s[:, 31] |= 1
    return s, [int.from_bytes(r.tobytes(), "big") for r in s]


def be32(ks):
    return np.frombuffer(b"".join((k % R).to_bytes(32, "big") for k in ks), dtype=np.uint8)


def check_same(*vs):
    for v in vs[1:]:
        assert np.asarray(v).tobytes() == np.asarray(vs[0]).tobytes(), "the calls compared disagree"


def alternate(calls, reps):
    """calls: name -> f() returning what must agree across the calls; medians of wall-clock ms after one warm-up each"""
    outs = {k: f() for k, f in calls.items()}
    check_same(*outs.values())
    t = {k: [] for k in calls}
    for _ in range(reps):
        for k, f in calls.items():
            r, ms = timed(f)
            check_same(r, outs[k])
            t[k].append(round(ms, 2))
    res = {k: {"ms": v, "median_ms": round(statistics.median(v), 2)} for k, v in t.items()}
    print(" | ".join(f"{k} {res[k]['median_ms']:.1f} ms" for k in calls), flush=True)
    return res, outs


def key_set(eng, B, impl, n, rng):
    sec, ints = secrets(rng, n)
    kb = eng.testdata_sign(impl, 0, sec.reshape(-1), *B.pack_messages([b""] * n))[0]
    return kb, ints


def sets_of(rng, q, size, n):
    idx = np.concatenate([rng.choice(n, size, replace=False) for _ in range(q)]).astype(np.uint32)
    return idx, np.arange(q + 1, dtype=np.uint64) * size


def multisigs(eng, impl, scheme, ints, idx, koff, qm, qoff):
    """the valid multi-signatures and the multi keys of every set"""
    q = koff.size - 1
    sums = [sum(ints[i] for i in idx[int(koff[j]):int(koff[j + 1])].tolist()) for j in range(q)]
    pks, sigs = eng.testdata_sign(impl, scheme, be32(sums), qm, qoff)
    return pks, sigs


def sum_stage(eng, impl, members, ms, peak):
    macs = members * FP_MUL[2 if impl == 1 else 1] * 300   # the keys of G2Impl are in G1, those of G1Impl in G2
    return {"decode_pk_stage_ms": round(ms, 3), "members": members, "algorithmic_mac": macs,
            "imad_peak_share": round(macs / (ms * 1e-3) / peak, 4) if ms > 0 else None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    import blsful_b200 as B
    eng = B.Engine([0])
    peak = eng.imad_peak()
    res = {"device": device_info(), "imad_peak_mac_per_s": peak, "shapes": {}}
    print(res["device"], f"IMAD peak {peak:.3e} MAC/s", flush=True)
    rng = np.random.default_rng(20261021)
    S = res["shapes"]
    qm = rng.integers(0, 256, size=(Q, 32), dtype=np.uint8)
    qm[:, :8] = np.arange(Q, dtype=np.uint64).view(np.uint8).reshape(Q, 8)
    qmf, qoff = qm.reshape(-1), np.arange(Q + 1, dtype=np.uint64) * 32

    # ---- A: 10,000 x 400 from a 2^16-key set, G2Impl and G1Impl ---------------------------------------------------------------
    for impl, name in ((2, "A"), (1, "A1")):
        pl, sl, pkg = B.pk_len(impl), B.sig_len(impl), (1 if impl == 2 else 2)
        kb, ints = key_set(eng, B, impl, KEYS, rng)
        idx, koff = sets_of(rng, Q, MEM, KEYS)
        agg_pk, sigs = multisigs(eng, impl, 2, ints, idx, koff, qmf, qoff)
        pk = kb.reshape(KEYS, pl)[idx].reshape(-1)
        ks = eng.key_set(impl, kb)
        keyed = lambda: eng.verify_multisig_batch_keyed_packed(ks, 2, koff, idx, sigs, qmf, qoff)
        calls = {"keyed": keyed, "unkeyed": lambda: eng.verify_multisig_batch_packed(impl, 2, koff, pk, sigs, qmf, qoff)}
        r, outs = alternate(calls, args.reps)
        assert outs["keyed"].tolist() == [0] * Q
        keyed()
        r["keyed_stage_ms"] = eng.last_stage_ms()
        r["sum_stage"] = sum_stage(eng, impl, Q * MEM, r["keyed_stage_ms"]["decode_pk"], peak)
        if impl == 2:
            # the present workaround: one blsgpu_sum_points per set (the first 100 timed, per set), one blsgpu_verify_batch
            loop = []
            for j in range(100):
                s, ms = timed(lambda: eng.sum_points(pkg, pk[int(koff[j]) * pl:int(koff[j + 1]) * pl]))
                assert s == agg_pk[j * pl:(j + 1) * pl].tobytes()
                loop.append(ms)
            vb, _ = alternate({"verify_batch_on_sums": lambda: eng.verify_batch_packed(impl, 2, agg_pk, sigs, qmf, qoff)}, args.reps)
            per_set = statistics.median(loop)
            r["workaround"] = {"sum_points_per_set_median_ms": round(per_set, 3), "verify_batch_ms": vb["verify_batch_on_sums"],
                               "total_estimate_ms": round(per_set * Q + vb["verify_batch_on_sums"]["median_ms"], 1)}
            print(f"{name} workaround: {per_set:.3f} ms per sum_points x {Q} + verify_batch", flush=True)
            # keyed verify_secure on the same quorums, with its own (weighted) aggregates
            sec_ints = ints
            member = np.empty(Q * MEM * sl, dtype=np.uint8)
            sec_rows = np.frombuffer(be32(sec_ints), dtype=np.uint8).reshape(KEYS, 32)
            for lo in range(0, Q * MEM, 1 << 20):
                hi = min(Q * MEM, lo + (1 << 20))
                o = np.arange(hi - lo + 1, dtype=np.uint64) * 32
                member[lo * sl:hi * sl] = eng.testdata_sign(impl, 2, sec_rows[idx[lo:hi]].reshape(-1),
                                                            np.ascontiguousarray(qm[np.arange(lo, hi) // MEM]).reshape(-1), o)[1]
            st, secure_aggs = eng.aggregate_secure_batch_keyed_packed(ks, koff, idx, member)
            assert int(st.max()) == 0
            del member
            vs, _ = alternate({"verify_secure_keyed": lambda: eng.verify_secure_batch_keyed_packed(ks, 2, koff, idx, secure_aggs, qmf, qoff),
                               "multisig_keyed": keyed}, args.reps)
            r["verify_secure_keyed_same_quorums"] = vs
            # D: the failure path
            for bad in (1, 100):
                pos = np.sort(rng.choice(Q, bad, replace=False))
                wrong = sigs.reshape(Q, sl).copy()
                wrong[pos] = sigs.reshape(Q, sl)[(pos + 1) % Q]
                wrong = wrong.reshape(-1)
                d, outs_d = alternate({"keyed": lambda: eng.verify_multisig_batch_keyed_packed(ks, 2, koff, idx, wrong, qmf, qoff),
                                       "unkeyed": lambda: eng.verify_multisig_batch_packed(impl, 2, koff, pk, wrong, qmf, qoff)}, args.reps)
                assert np.nonzero(outs_d["keyed"])[0].tolist() == pos.tolist()
                S[f"D_{bad}_wrong"] = d
        ks.close()
        S[name] = r

    # ---- B: one multi-signature of 2^20 signers ------------------------------------------------------------------------------
    n = 1 << 20
    kb, ints = key_set(eng, B, 2, n, rng)
    idx = np.arange(n, dtype=np.uint32)
    koff = np.array([0, n], dtype=np.uint64)
    agg_pk, sig = multisigs(eng, 2, 2, ints, idx, koff, qmf[:32], qoff[:2])
    ks = eng.key_set(2, kb)

    def sum_then_verify():
        s = eng.sum_points(1, kb)
        return eng.verify_batch(2, 2, [s], [sig.tobytes()], [qm[0].tobytes()])
    r, outs = alternate({"keyed": lambda: eng.verify_multisig_batch_keyed_packed(ks, 2, koff, idx, sig, qmf[:32], qoff[:2]),
                         "sum_points_then_verify_batch": sum_then_verify}, args.reps)
    assert outs["keyed"].tolist() == [0]
    eng.verify_multisig_batch_keyed_packed(ks, 2, koff, idx, sig, qmf[:32], qoff[:2])
    r["keyed_stage_ms"] = eng.last_stage_ms()
    r["sum_stage"] = sum_stage(eng, 2, n, r["keyed_stage_ms"]["decode_pk"], peak)
    S["B"] = r
    ks.close()

    # ---- C: 2^18 sets x 2 signers --------------------------------------------------------------------------------------------
    q = 1 << 18
    kb, ints = key_set(eng, B, 2, KEYS, rng)
    idx, koff = sets_of(rng, q, 2, KEYS)
    cm = rng.integers(0, 256, size=(q, 32), dtype=np.uint8).reshape(-1)
    coff = np.arange(q + 1, dtype=np.uint64) * 32
    agg_pk, sigs = multisigs(eng, 2, 2, ints, idx, koff, cm, coff)
    ks = eng.key_set(2, kb)
    keyed = lambda: eng.verify_multisig_batch_keyed_packed(ks, 2, koff, idx, sigs, cm, coff)
    r, outs = alternate({"keyed": keyed, "verify_batch_on_sums": lambda: eng.verify_batch_packed(2, 2, agg_pk, sigs, cm, coff)}, args.reps)
    assert outs["keyed"].tolist() == [0] * q
    keyed()
    r["keyed_stage_ms"] = eng.last_stage_ms()
    r["sum_stage"] = sum_stage(eng, 2, 2 * q, r["keyed_stage_ms"]["decode_pk"], peak)
    S["C"] = r
    ks.close()

    # ---- E: blsgpu_sum_points_batch over 10,000 x 400 signatures --------------------------------------------------------------
    sec, _ = secrets(rng, KEYS)
    pts = eng.testdata_sign(2, 0, sec.reshape(-1), *B.pack_messages([b"E"] * KEYS))[1]
    idx, soff = sets_of(rng, Q, MEM, KEYS)
    flat = pts.reshape(KEYS, 96)[idx].reshape(-1)
    (st, bad, sums), ms = timed(lambda: eng.sum_points_batch_packed(2, soff, flat))
    r, outs = alternate({"sum_points_batch": lambda: eng.sum_points_batch_packed(2, soff, flat)[2]}, args.reps)
    loop = []
    for j in range(100):
        s, t = timed(lambda: eng.sum_points(2, flat[int(soff[j]) * 96:int(soff[j + 1]) * 96]))
        assert s == sums[j * 96:(j + 1) * 96].tobytes()
        loop.append(t)
    r["sum_points_per_set_median_ms"] = round(statistics.median(loop), 3)
    r["loop_total_estimate_ms"] = round(statistics.median(loop) * Q, 1)
    S["E"] = r
    print(f"E loop: {statistics.median(loop):.3f} ms per set", flush=True)

    res["status_vectors_identical"] = True
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "verify_multisig_b200.json"), "w") as f:
        json.dump(res, f, indent=1)
    eng.close()


if __name__ == "__main__":
    main()

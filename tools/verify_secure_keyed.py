#!/usr/bin/env python
"""Measures the keyed secure-aggregation calls (quorum members named by index into a key set) against the unkeyed calls on
the same quorums, the split of the unkeyed cfg-5 call, and the one-time cost of a key set's secure view.

Shapes (Bls12381G2Impl, Basic; quorum j signs a 32-byte message; member sigs from blsgpu_testdata_sign):
  split      the unkeyed blsgpu_verify_secure_batch at 10,000 x 400 over 4M distinct keys (Modern), under torch.profiler in a
             pass of its own: host plan = from the start of the call to its first host-to-device copy (the host sort of
             make_secure_plan, argument checks and arena sizing), upload = the device time of its host-to-device copies,
             key decode / signature decode = k_decode + k_subgroup_check of the key / signature group, MSM = k_secure_* +
             k_to_affine, verify = every other kernel; plus blsgpu_last_stage_ms of a call without the profiler
  4M         keyed (a 4M-key set, member i = key i) against unkeyed, Modern and Legacy: verify accepted, verify with two
             swapped signatures, aggregate; alternated --reps times after a warm-up of each
  4096       keyed over a 4,096-key set (400 distinct members per quorum drawn from it) against unkeyed on the written-out keys
  view       the first keyed call on a new set in each format minus the same call once the view exists, for 4,096, 2^20 and
             4M keys
Wall clock around each call (every call ends in a stream synchronisation).  Status vectors and aggregate bytes of keyed and
unkeyed calls must be identical in every shape; the tool stops otherwise.

    python tools/verify_secure_keyed.py --out DIR [--reps 3] [--quorums 10000]   -> DIR/verify_secure_keyed_b200.json
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

MEM = 400


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
    return s


def sign_members(eng, sec, idx, qm, chunk=1 << 20):
    """member sigs: key idx[i] signs its quorum's message qm[i // MEM]"""
    tot = idx.size
    out = np.empty(tot * 96, dtype=np.uint8)
    for lo in range(0, tot, chunk):
        hi = min(tot, lo + chunk)
        o = np.arange(hi - lo + 1, dtype=np.uint64) * 32
        out[lo * 96:hi * 96] = eng.testdata_sign(2, 0, sec[idx[lo:hi]].reshape(-1), np.ascontiguousarray(qm[np.arange(lo, hi) // MEM]).reshape(-1), o)[1]
    return out


def set_keys(eng, B, sec):
    return eng.testdata_sign(2, 0, sec.reshape(-1), *B.pack_messages([b""] * sec.shape[0]))[0]


def split_unkeyed(eng, koff, pk, aggs, qm, qoff):
    import torch
    from torch.profiler import ProfilerActivity, profile, record_function
    call = lambda: eng.verify_secure_batch_packed(2, 0, koff, pk, aggs, qm, qoff, 1)
    call()
    _, wall = timed(call)
    stages = eng.last_stage_ms()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        with record_function("verify_secure_call"):
            call()
        torch.cuda.synchronize()
    ev = prof.events()
    rng_ev = [e for e in ev if e.name == "verify_secure_call"][0]
    t0 = rng_ev.time_range.start
    copies = sorted(e.time_range.start for e in ev if e.name == "cudaMemcpyAsync" and e.time_range.start >= t0)
    cat = {"upload": 0.0, "key_decode": 0.0, "sig_decode": 0.0, "msm": 0.0, "verify": 0.0}
    kernels = {}
    for e in ev:
        if e.device_type.name != "CUDA" or e.name == "verify_secure_call":   # the annotation's own span on the device
            continue
        ms = (e.time_range.end - e.time_range.start) / 1e3
        n = e.name
        kernels[n[:120]] = kernels.get(n[:120], 0.0) + ms
        if "Memcpy HtoD" in n:
            cat["upload"] += ms
        elif "Memcpy" in n or "Memset" in n:
            continue
        elif "k_decode" in n or "k_subgroup_check" in n:
            cat["sig_decode" if "Fp2" in n else "key_decode"] += ms   # G2Impl: keys in G1 (Fp), signatures in G2 (Fp2)
        elif "k_secure" in n or "k_to_affine<" in n or "k_to_affineIN" in n:
            cat["msm"] += ms
        else:
            cat["verify"] += ms
    cat["host_plan"] = (copies[0] - t0) / 1e3 if copies else None
    return {"wall_ms_no_profiler": wall, "stage_ms": stages, "profiled_ms": {k: round(v, 2) for k, v in cat.items() if v is not None},
            "profiled_device_ms_by_name": {k: round(v, 2) for k, v in sorted(kernels.items(), key=lambda kv: -kv[1])}}


def ab(name, keyed, unkeyed, reps, check):
    rk, ru = keyed(), unkeyed()   # warm-up (and, for keyed, the secure view)
    check(rk, ru)
    tk, tu = [], []
    for _ in range(reps):
        r, t = timed(unkeyed)
        tu.append(t)
        r2, t2 = timed(keyed)
        tk.append(t2)
        check(r2, r)
    mk, mu = statistics.median(tk), statistics.median(tu)
    print(f"{name}: keyed {mk:.1f} ms, unkeyed {mu:.1f} ms, ratio {mu / mk:.2f}", flush=True)
    return {"keyed_ms": [round(t, 1) for t in tk], "unkeyed_ms": [round(t, 1) for t in tu], "keyed_median_ms": round(mk, 1),
            "unkeyed_median_ms": round(mu, 1), "unkeyed_over_keyed": round(mu / mk, 3)}


def same_status(a, b):
    assert a.tolist() == b.tolist(), "keyed and unkeyed statuses differ"


def same_agg(a, b):
    assert a[0].tolist() == b[0].tolist() and a[1].tobytes() == b[1].tobytes(), "keyed and unkeyed aggregates differ"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--quorums", type=int, default=10_000)
    args = ap.parse_args()
    import blsful_b200 as B
    eng = B.Engine([0])
    res = {"device": device_info(), "quorums": args.quorums, "members": MEM}
    print(res["device"], flush=True)
    rng = np.random.default_rng(20261021)
    q = args.quorums
    tot = q * MEM
    qm = rng.integers(0, 256, size=(q, 32), dtype=np.uint8)
    qm[:, :8] = np.arange(q, dtype=np.uint64).view(np.uint8).reshape(q, 8)
    koff = np.arange(q + 1, dtype=np.uint64) * MEM
    qoff = np.arange(q + 1, dtype=np.uint64) * 32
    qmf = qm.reshape(-1)

    # 4M distinct keys, member i = key i
    sec = secrets(rng, tot)
    idx = np.arange(tot, dtype=np.uint32)
    member = sign_members(eng, sec, idx, qm)
    kb = set_keys(eng, B, sec)
    st, aggs = eng.aggregate_secure_batch_packed(2, koff, kb, member)
    assert int(st.max()) == 0
    res["split_unkeyed_modern"] = split_unkeyed(eng, koff, kb, aggs, qmf, qoff)
    print("split", res["split_unkeyed_modern"], flush=True)

    res["shapes"] = {}
    enc = {1: (kb, member, aggs)}
    pk_l, mem_l = eng.recode_points_packed(1, kb, 1, 0), eng.recode_points_packed(2, member, 1, 0)
    st, aggs_l = eng.aggregate_secure_batch_packed(2, koff, pk_l, mem_l, 0)   # Legacy hashes the keys' Legacy bytes
    assert int(st.max()) == 0
    enc[0] = (pk_l, mem_l, aggs_l)
    for fmt, fname in ((1, "modern"), (0, "legacy")):
        pk_f, mem_f, agg_f = enc[fmt]
        ks = eng.key_set(2, pk_f, fmt)
        swapped = agg_f.copy().reshape(q, 96)
        swapped[[3, 4]] = swapped[[4, 3]]
        swapped = swapped.reshape(-1)
        r = res["shapes"]
        r[f"4M_verify_{fname}"] = ab(f"4M verify {fname}", lambda: eng.verify_secure_batch_keyed_packed(ks, 0, koff, idx, agg_f, qmf, qoff, fmt),
                                      lambda: eng.verify_secure_batch_packed(2, 0, koff, pk_f, agg_f, qmf, qoff, fmt), args.reps, same_status)
        r[f"4M_verify_two_swapped_{fname}"] = ab(
            f"4M verify two swapped {fname}", lambda: eng.verify_secure_batch_keyed_packed(ks, 0, koff, idx, swapped, qmf, qoff, fmt),
            lambda: eng.verify_secure_batch_packed(2, 0, koff, pk_f, swapped, qmf, qoff, fmt), args.reps, same_status)
        assert np.nonzero(eng.verify_secure_batch_keyed_packed(ks, 0, koff, idx, swapped, qmf, qoff, fmt))[0].tolist() == [3, 4]
        r[f"4M_aggregate_{fname}"] = ab(f"4M aggregate {fname}", lambda: eng.aggregate_secure_batch_keyed_packed(ks, koff, idx, mem_f, fmt),
                                         lambda: eng.aggregate_secure_batch_packed(2, koff, pk_f, mem_f, fmt), args.reps, same_agg)
        assert eng.aggregate_secure_batch_keyed_packed(ks, koff, idx, mem_f, fmt)[1].tobytes() == agg_f.tobytes()
        ks.close()
    del enc

    # realistic shape: 400 distinct members per quorum from a 4,096-key set
    sec4 = secrets(rng, 4096)
    idx4 = np.concatenate([rng.choice(4096, MEM, replace=False) for _ in range(q)]).astype(np.uint32)
    member4 = sign_members(eng, sec4, idx4, qm)
    kb4 = set_keys(eng, B, sec4)
    pk4 = kb4.reshape(4096, 48)[idx4].reshape(-1)
    ks4 = eng.key_set(2, kb4)
    st4, agg4 = eng.aggregate_secure_batch_keyed_packed(ks4, koff, idx4, member4)
    assert int(st4.max()) == 0
    r = res["shapes"]
    r["4096_verify_modern"] = ab("4096-key set verify", lambda: eng.verify_secure_batch_keyed_packed(ks4, 0, koff, idx4, agg4, qmf, qoff),
                                 lambda: eng.verify_secure_batch_packed(2, 0, koff, pk4, agg4, qmf, qoff), args.reps, same_status)
    r["4096_aggregate_modern"] = ab("4096-key set aggregate", lambda: eng.aggregate_secure_batch_keyed_packed(ks4, koff, idx4, member4),
                                    lambda: eng.aggregate_secure_batch_packed(2, koff, pk4, member4), args.reps, same_agg)
    ks4.close()

    # one-time cost of the secure view: the first keyed call in a format minus the same call once its view exists
    res["view_build_ms"] = {}
    one = np.array([0, 1], dtype=np.uint64)
    for n in (4096, 1 << 20, tot):
        keys = np.tile(kb, -(-n * 48 // kb.size))[:n * 48]
        ks = eng.key_set(2, keys)
        for fmt, fname in ((1, "modern"), (0, "legacy")):
            call = lambda: eng.aggregate_secure_batch_keyed_packed(ks, one, np.zeros(1, dtype=np.uint32), enc_member(eng, member[:96], fmt), fmt)
            _, first = timed(call)
            later = statistics.median([timed(call)[1] for _ in range(3)])
            res["view_build_ms"][f"{n}_{fname}"] = round(first - later, 1)
            print(f"view {n} {fname}: {first - later:.1f} ms", flush=True)
        ks.close()
    res["status_and_bytes_identical"] = True
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "verify_secure_keyed_b200.json"), "w") as f:
        json.dump(res, f, indent=1)
    eng.close()


def enc_member(eng, sig, fmt):
    return sig if fmt == 1 else eng.recode_points_packed(2, sig, 1, 0)


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""Measures changing a 2^20-key set in place (blsgpu_keyset_update / blsgpu_keyset_append) against re-creating it.

For each impl, a set of 2^20 distinct keys, with no secure view, with the Modern view, and (Bls12381G2Impl, the only impl
with Legacy secure calls) with both views:
  update k   blsgpu_keyset_update of k = 1, 1,000 and 65,536 keys (distinct random indices; the calls alternate between new
             keys and the original ones, so that every call changes k keys)
  append     blsgpu_keyset_append of 1,000 keys (each call grows the set by 1,000 keys)
and, against them:
  create     blsgpu_keyset_create of the same 2^20 keys
  view       the extra wall clock of the first keyed secure call in a format (which builds that view) over the second
             (aggregate_secure over one quorum of 3 keys)
Each number is the median wall clock of --reps calls; every call ends in its own stream synchronisation.  The card's name,
power limit and maximum SM clock are read in the same run.

    python tools/keyset_update.py --out DIR [--reps 5]     -> DIR/keyset_update_b200.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "agora-blsful_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)
sys.dont_write_bytecode = True

import numpy as np

N = 1 << 20
KS = (1, 1000, 65536)
APPEND = 1000


def device_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"unavailable: {e}"


def timed(fn):
    t = time.perf_counter()
    out = fn()
    return (time.perf_counter() - t) * 1e3, out


def median(xs):
    return float(np.median(np.array(xs)))


_KEYS = {}


def keys(eng, B, impl, count, seed):
    if (impl, count, seed) in _KEYS:
        return _KEYS[(impl, count, seed)]
    rng = np.random.default_rng(seed)
    secret = np.zeros((count, 32), dtype=np.uint8)
    secret[:, 8:] = rng.integers(0, 256, size=(count, 24), dtype=np.uint8)
    secret[:, 31] |= 1
    pk, sg = eng.testdata_sign(impl, 0, secret.reshape(-1), np.zeros(0, dtype=np.uint8), np.zeros(count + 1, dtype=np.uint64))
    _KEYS[(impl, count, seed)] = pk.reshape(count, B.pk_len(impl)), sg.reshape(count, B.sig_len(impl))
    return _KEYS[(impl, count, seed)]


def run(eng, B, impl, views, reps):
    from oracle import bls_oracle as O
    base, member = keys(eng, B, impl, N, 100 + impl)
    new, _ = keys(eng, B, impl, max(KS) + APPEND * (reps + 1), 200 + impl)
    rng = np.random.default_rng(7)
    quorum = (np.array([0, 3], dtype=np.uint64), np.array([5, 1, 2], dtype=np.uint32))
    fmts = [O.MODERN, O.LEGACY][:views]

    def secure(ks, fmt):
        sg = np.ascontiguousarray(member[quorum[1]]).reshape(-1)
        if fmt == O.LEGACY:
            sg = eng.recode_points_packed(impl, sg, O.MODERN, O.LEGACY)   # the signature group's number is the impl's
        st, _ = eng.aggregate_secure_batch_keyed_packed(ks, quorum[0], quorum[1], sg, fmt)
        assert st.tolist() == [0]

    res = {"impl": impl, "views": views}
    create = []
    for _ in range(reps):
        ms, ks = timed(lambda: eng.key_set(impl, base.reshape(-1)))
        create.append(ms)
        if len(create) < reps:
            ks.close()
    res["create_ms"] = median(create)
    view_ms = {}
    for fmt in fmts:
        first, _ = timed(lambda: secure(ks, fmt))
        second = median([timed(lambda: secure(ks, fmt))[0] for _ in range(reps)])
        view_ms["modern" if fmt == O.MODERN else "legacy"] = first - second
    res["view_build_ms"] = view_ms
    for k in KS:
        idx = rng.permutation(N)[:k].astype(np.uint32)
        changed, original = np.ascontiguousarray(new[:k]).reshape(-1), np.ascontiguousarray(base[idx]).reshape(-1)
        eng.update_key_set(ks, idx, changed)   # warm-up (and sizes the scratch)
        eng.update_key_set(ks, idx, original)
        times = []
        for r in range(reps):
            ms, st = timed(lambda: eng.update_key_set(ks, idx, changed if r % 2 == 0 else original))
            assert not st.any()
            times.append(ms)
        if reps % 2:
            eng.update_key_set(ks, idx, original)
        res[f"update_{k}_ms"] = median(times)
    times = []
    for r in range(reps + 1):
        chunk = np.ascontiguousarray(new[max(KS) + APPEND * r:max(KS) + APPEND * (r + 1)]).reshape(-1)
        ms, st = timed(lambda: eng.append_key_set(ks, chunk))
        assert not st.any()
        if r:   # the first append warms the kernels and the scratch up
            times.append(ms)
    res[f"append_{APPEND}_ms"] = median(times)
    for fmt in fmts:   # the views still serve the keyed secure calls
        secure(ks, fmt)
    assert len(ks) == N + APPEND * (reps + 1)
    ks.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    import blsful_b200 as B
    eng = B.Engine([0])
    out = {"device": device_info(), "n": N, "reps": args.reps,
           "method": "median wall clock of --reps calls, each ending in its own stream synchronisation", "runs": []}
    for impl in (2, 1):
        for views in ((0, 1, 2) if impl == 2 else (0, 1)):
            r = run(eng, B, impl, views, args.reps)
            print(json.dumps(r), flush=True)
            out["runs"].append(r)
    out["device_after"] = device_info()
    eng.close()
    path = os.path.join(args.out, "keyset_update_b200.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", path)


if __name__ == "__main__":
    main()

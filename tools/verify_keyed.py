#!/usr/bin/env python
"""Measures the keyed verify calls (keys decoded once into a key set, named by index) against the unkeyed calls on the same
items, and the cost of creating a key set.

Shapes (2^20 items; message of an item or of a group = SHA-256 of its index, 32 bytes):
  V2, V1  blsgpu_verify_batch[_keyed], distinct messages and keys (a 2^20-key set), Bls12381G2Impl / Bls12381G1Impl
  GA, GB  blsgpu_verify_batch_grouped[_keyed], G2Impl, every item its own key, over 1 / 1,000 messages (DESIGN.md section 6)
  S1, S1000  1,000 messages signed by keys of a 2^16-key set (each key signs ~16 items), G2Impl, with 1 / 1,000 bad items
          (another item's signature): both pairs of calls
  create  blsgpu_keyset_create of 2^20 keys of each group
Every shape warms both calls up once, then alternates keyed / unkeyed --reps times.  Wall clock around the call (it ends in a
stream synchronisation), the stage and kernel times of the last call of each kind.  The status vectors of the two calls must
be byte-identical and equal the plant.  `saving_over_decode_pk` = (unkeyed - keyed median wall clock) / the unkeyed call's
decode_pk stage time in the same run.

    python tools/verify_keyed.py --out DIR [--shapes V2,GA] [--reps 3]     -> DIR/verify_keyed.json
"""
import argparse
import hashlib
import json
import os
import random
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


def device_info():
    info = {}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["nvidia_smi"] = out
    except Exception as e:  # noqa: BLE001
        info["nvidia_smi"] = f"unavailable: {e}"
    return info


def hashed(tag, count):
    return np.frombuffer(b"".join(hashlib.sha256(b"%s/%d" % (tag, j)).digest() for j in range(count)), dtype=np.uint8).reshape(count, 32)


def make_shape(eng, B, rnd, impl, q, nkeys):
    """N items over q messages (q = N: every item its own message) and nkeys keys (item i: message idx[i], key kidx[i])"""
    nrng = np.random.default_rng(q * 7 + nkeys)
    idx = np.arange(N, dtype=np.uint32) if q == N else nrng.integers(0, q, size=N, dtype=np.uint32)
    kidx = np.arange(N, dtype=np.uint32) if nkeys == N else nrng.integers(0, nkeys, size=N, dtype=np.uint32)
    msgs = hashed(b"keyed/%d" % q, q)
    secret = np.frombuffer(b"".join(rnd.randrange(1, 2 ** 250).to_bytes(32, "big") for _ in range(nkeys)), dtype=np.uint8).reshape(nkeys, 32)
    data_items = np.ascontiguousarray(msgs[idx]).reshape(-1)
    off_items = np.arange(N + 1, dtype=np.uint64) * np.uint64(32)
    pk, sg = eng.testdata_sign(impl, 0, np.ascontiguousarray(secret[kidx]).reshape(-1), data_items, off_items)
    L = B.pk_len(impl)
    if nkeys == N:
        keys = pk
    else:   # the key of key index k, from the first item that has it (every index of the set has one at these sizes)
        first = np.full(nkeys, -1, dtype=np.int64)
        first[kidx[::-1]] = np.arange(N - 1, -1, -1)
        assert (first >= 0).all()
        keys = np.ascontiguousarray(pk.reshape(N, L)[first]).reshape(-1)
    return dict(impl=impl, q=q, idx=idx, kidx=kidx, keys=keys, pk=pk, sg=sg, data=np.ascontiguousarray(msgs).reshape(-1),
                off=np.arange(q + 1, dtype=np.uint64) * np.uint64(32), data_items=data_items, off_items=off_items)


def calls(kind):
    if kind == "batch":
        return (("keyed", lambda e, ks, s: e.verify_batch_keyed_packed(ks, 0, s["kidx"], s["sg"], s["data_items"], s["off_items"])),
                ("unkeyed", lambda e, ks, s: e.verify_batch_packed(s["impl"], 0, s["pk"], s["sg"], s["data_items"], s["off_items"])))
    return (("keyed", lambda e, ks, s: e.verify_batch_grouped_keyed_packed(ks, 0, s["kidx"], s["sg"], s["idx"], s["data"], s["off"])),
            ("unkeyed", lambda e, ks, s: e.verify_batch_grouped_packed(s["impl"], 0, s["pk"], s["sg"], s["idx"], s["data"], s["off"])))


def measure(B, s, kind, reps, bad):
    eng = B.Engine([0])
    ks = eng.key_set(s["impl"], s["keys"])
    assert not ks.status.any()
    out, res = {}, {}
    for name, fn in calls(kind):
        res[name] = fn(eng, ks, s)  # warm-up
        out[name] = dict(wall_ms=[])
    for _ in range(reps):
        for name, fn in calls(kind):
            t0 = time.perf_counter()
            st = fn(eng, ks, s)
            out[name]["wall_ms"].append((time.perf_counter() - t0) * 1e3)
            out[name]["stage_ms"] = eng.last_stage_ms()
            out[name]["kernel_ms"] = {k: [round(ms, 3), c] for k, (ms, c) in eng.last_kernel_ms().items()}
            assert st.tobytes() == res[name].tobytes()
    eng.close()
    assert res["keyed"].tobytes() == res["unkeyed"].tobytes()
    assert np.flatnonzero(res["keyed"]).tolist() == bad
    for name in ("keyed", "unkeyed"):
        out[name]["wall_ms_median"] = float(np.median(out[name]["wall_ms"]))
    saved = out["unkeyed"]["wall_ms_median"] - out["keyed"]["wall_ms_median"]
    out["saved_ms"] = saved
    out["unkeyed_decode_pk_ms"] = out["unkeyed"]["stage_ms"]["decode_pk"]
    out["saving_over_decode_pk"] = saved / out["unkeyed_decode_pk_ms"]
    return out


def plant(s, bad):
    L = s["sg"].size // N
    sg = s["sg"].reshape(N, L).copy()
    for i in bad:
        sg[i] = s["sg"].reshape(N, L)[(i + 1) % N]
    return dict(s, sg=sg.reshape(-1))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--shapes", default="create,V2,V1,GA,GB,S1,S1000")
    a = ap.parse_args()
    import blsful_b200 as B
    os.makedirs(a.out, exist_ok=True)
    wanted = a.shapes.split(",")
    eng = B.Engine([0])
    rnd = random.Random(20261020)
    res = {"info": device_info(), "scheme": "Basic", "format": "Modern", "rlc_bits": 64, "items": N, "shapes": {}}

    def emit(name, r):
        res["shapes"][name] = r
        print(name, json.dumps(r), flush=True)
        with open(os.path.join(a.out, "verify_keyed.json"), "w") as f:
            json.dump(res, f, indent=1)

    if "create" in wanted:
        for impl in (2, 1):
            keys = make_shape(eng, B, rnd, impl, N, N)["pk"]
            e = B.Engine([0])
            e.key_set(impl, keys[:B.pk_len(impl) * 4096]).close()   # warm-up
            ms = []
            for _ in range(a.reps):
                t0 = time.perf_counter()
                ks = e.key_set(impl, keys)
                ms.append((time.perf_counter() - t0) * 1e3)
                assert not ks.status.any()
                ks.close()
            e.close()
            emit("create_g%d" % (1 if impl == 2 else 2), dict(impl=impl, keys=N, wall_ms=ms, wall_ms_median=float(np.median(ms))))
    for name, impl, kind, q, nkeys in (("V2", 2, "batch", N, N), ("V1", 1, "batch", N, N), ("GA", 2, "grouped", 1, N),
                                       ("GB", 2, "grouped", 1000, N)):
        if name in wanted:
            s = make_shape(eng, B, rnd, impl, q, nkeys)
            emit(name, dict(impl=impl, call=kind, q=q, keys=nkeys, bad=0, **measure(B, s, kind, a.reps, [])))
    if "S1" in wanted or "S1000" in wanted:
        s = make_shape(eng, B, rnd, 2, 1000, 1 << 16)
        for nbad in (1, 1000):
            if "S%d" % nbad not in wanted:
                continue
            bad = sorted(random.Random(nbad).sample(range(N), nbad))
            p = plant(s, bad)
            for kind in ("grouped", "batch"):
                emit("S%d_%s" % (nbad, kind), dict(impl=2, call=kind, q=1000, keys=1 << 16, bad=nbad, **measure(B, p, kind, a.reps, bad)))
    eng.close()


if __name__ == "__main__":
    main()

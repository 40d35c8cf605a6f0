#!/usr/bin/env python
"""Measures blsgpu_aggregate_verify_batch against a loop of single blsgpu_aggregate_verify calls (Bls12381G2Impl, Basic).

Shapes (q aggregates x pairs each):
  A  1,000 x 100          many mid-sized aggregates (a block's worth)
  B  1 x 100,000          one large aggregate (cfg 4's shape)
  C  10,000 x 2           tiny aggregates: each fills one Miller group of 6 slots, 2/3 of them padding
  D  shape A with 1 wrong aggregate, and with 100 (the failure search)
The batch call is warmed up once and timed over --reps calls (wall clock around the call, which ends in a stream
synchronisation; device time = sum of blsgpu_last_stage_ms).  The loop times --loop real single calls (shape B: the one
aggregate, --loop times) and reports what it timed; nothing is extrapolated.  Shape C repeats 500
distinct aggregates 20 times (the work per aggregate does not depend on which one it is).

    python tools/agg_verify_batch.py --out DIR      -> DIR/agg_verify_batch.json
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


def device_info():
    info = {}
    try:
        import torch
        info["device"] = torch.cuda.get_device_name(0)
    except Exception as e:  # noqa: BLE001
        info["device"] = f"unavailable: {e}"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["nvidia_smi"] = out
    except Exception as e:  # noqa: BLE001
        info["nvidia_smi"] = f"unavailable: {e}"
    return info


def make_aggregates(eng, B, rnd, q, n, tag):
    """q distinct valid aggregates of n pairs: flat pk / message buffers, set offsets and q signatures."""
    msgs = [hashlib.sha256(b"%s/%d" % (tag, i)).digest() for i in range(q * n)]
    k = np.frombuffer(b"".join(rnd.randrange(1, 2 ** 250).to_bytes(32, "big") for _ in range(q * n)), dtype=np.uint8)
    data, off = B.pack_messages(msgs)
    pks, sigs = eng.testdata_sign(2, 0, k, data, off)
    agg = b"".join(eng.sum_points(2, sigs[j * n * 96:(j + 1) * n * 96]) for j in range(q))
    soff = np.arange(q + 1, dtype=np.uint64) * np.uint64(n)
    return dict(q=q, n=n, soff=soff, pk=pks, data=data, off=off, sg=np.frombuffer(agg, dtype=np.uint8).copy())


def tile(s, times):
    q, n = s["q"], s["n"]
    data = np.tile(s["data"], times)
    step = np.uint64(s["off"][-1])
    off = np.concatenate([s["off"][:1]] + [s["off"][1:] + step * np.uint64(t) for t in range(times)])
    return dict(q=q * times, n=n, soff=np.arange(q * times + 1, dtype=np.uint64) * np.uint64(n), pk=np.tile(s["pk"], times), data=data,
                off=off, sg=np.tile(s["sg"], times))


def time_batch(eng, s, reps):
    st, _ = eng.aggregate_verify_batch_packed(2, 0, s["soff"], s["pk"], s["data"], s["off"], s["sg"])  # warm-up
    walls, dev = [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        st, _ = eng.aggregate_verify_batch_packed(2, 0, s["soff"], s["pk"], s["data"], s["off"], s["sg"])
        walls.append((time.perf_counter() - t0) * 1e3)
        dev.append(sum(eng.last_stage_ms().values()))
    return st, dict(wall_ms=walls, wall_ms_median=float(np.median(walls)), device_ms=dev, device_ms_median=float(np.median(dev)))


def time_loop(eng, s, calls):
    """`calls` single blsgpu_aggregate_verify calls over aggregates 0, 1, ... (modulo q), after one warm-up call."""
    n = s["n"]
    lib = eng._lib
    st = np.zeros(1, dtype=np.uint8)
    idx = np.full(2, -1, dtype=np.int64)
    statuses = []

    def one(j):
        lo, hi = j * n, (j + 1) * n
        off = np.ascontiguousarray(s["off"][lo:hi + 1] - s["off"][lo])
        data = s["data"][int(s["off"][lo]):int(s["off"][hi])]
        pk = s["pk"][lo * 48:hi * 48]
        sg = s["sg"][j * 96:(j + 1) * 96]
        rc = lib.blsgpu_aggregate_verify(eng._ctx, 2, 0, 1, n, pk.ctypes.data, data.ctypes.data, off.ctypes.data, sg.ctypes.data,
                                         st.ctypes.data, idx.ctypes.data)
        assert rc == 0, rc
        return int(st[0])

    one(0)
    t0 = time.perf_counter()
    for j in range(calls):
        statuses.append(one(j % s["q"]))
    total = (time.perf_counter() - t0) * 1e3
    return statuses, dict(calls=calls, total_ms=total, per_call_ms=total / calls)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--loop", type=int, default=100)
    a = ap.parse_args()
    import blsful_b200 as B
    os.makedirs(a.out, exist_ok=True)
    eng = B.Engine([0])
    rnd = random.Random(12345)
    res = {"info": device_info(), "impl": "Bls12381G2Impl", "scheme": "Basic", "format": "Modern", "rlc_bits": 64, "shapes": {}}
    A = make_aggregates(eng, B, rnd, 1000, 100, b"A")
    Bs = make_aggregates(eng, B, rnd, 1, 100_000, b"B")
    C = tile(make_aggregates(eng, B, rnd, 500, 2, b"C"), 20)
    shapes = [("A", A, []), ("B", Bs, []), ("C", C, [])]
    for nbad in (1, 100):
        bad = sorted(random.Random(nbad).sample(range(1000), nbad))
        D = dict(A, sg=A["sg"].copy())
        for j in bad:
            D["sg"][j * 96:(j + 1) * 96] = A["sg"][((j + 1) % 1000) * 96:((j + 1) % 1000 + 1) * 96]
        shapes.append(("D%d" % nbad, D, bad))
    for name, s, bad in shapes:
        st, batch = time_batch(eng, s, a.reps)
        assert [j for j in range(s["q"]) if st[j]] == bad and all(st[j] == 1 for j in bad), name
        calls = max(a.loop, 1)
        # shape B has one aggregate: it is verified `calls` times; otherwise aggregates 0 .. calls-1 (wrapping round)
        singles, loop = time_loop(eng, s, calls)
        assert singles == [int(st[j % s["q"]]) for j in range(calls)], name
        res["shapes"][name] = dict(q=s["q"], pairs_per_aggregate=s["n"], bad=len(bad), batch=batch, single_loop=loop)
        print(name, json.dumps(res["shapes"][name]), flush=True)
    eng.close()
    with open(os.path.join(a.out, "agg_verify_batch.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

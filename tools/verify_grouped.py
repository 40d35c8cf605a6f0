#!/usr/bin/env python
"""Measures blsgpu_verify_batch_grouped against blsgpu_verify_batch on the same 2^20 items (Bls12381G2Impl, Basic).

Shapes (items over q messages, each item a fresh key; message i = SHA-256 of its index, 32 bytes):
  A  q = 1              every item signs one message: 10,923 leaves of up to 96 items (the bucket kernel)
  B  q = 1,000          ~1,049 items per message
  C  q = 2^19           pairs: leaves of 2 items (the per-item kernel)
  D  q = 2^20           every message distinct: one leaf per item
  E  shape B with 1 and with 1,000 bad items (another item's signature) at seeded positions: the failure search
Each shape warms both calls up once, then alternates grouped / per-item --reps times.  Wall clock around the call (it
ends in a stream synchronisation), the stage and kernel times of the last call of each kind, and the device memory a
fresh context holds after one call while no other context holds an arena (its arena, which only grows: the call's
high-water mark).  The two status vectors
must be byte-identical and equal the plant.

    python tools/verify_grouped.py --out DIR [--shapes A,B] [--label L]     -> DIR/verify_grouped.json
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


def make_shape(eng, B, rnd, q):
    """N items over q messages (item i signs message idx[i]; every message has an item when q <= N / 2)"""
    idx = (np.arange(N, dtype=np.uint64) % np.uint64(q)).astype(np.uint32)
    idx = idx[np.random.default_rng(q).permutation(N)]
    msgs = np.frombuffer(b"".join(hashlib.sha256(b"grouped/%d/%d" % (q, j)).digest() for j in range(q)), dtype=np.uint8).reshape(q, 32)
    data_items = np.ascontiguousarray(msgs[idx]).reshape(-1)
    off_items = np.arange(N + 1, dtype=np.uint64) * np.uint64(32)
    keys = np.frombuffer(b"".join(rnd.randrange(1, 2 ** 250).to_bytes(32, "big") for _ in range(N)), dtype=np.uint8)
    pk, sg = eng.testdata_sign(2, 0, keys, data_items, off_items)
    return dict(q=q, idx=idx, data=np.ascontiguousarray(msgs).reshape(-1), off=np.arange(q + 1, dtype=np.uint64) * np.uint64(32),
                data_items=data_items, off_items=off_items, pk=pk, sg=sg)


def run_grouped(eng, s):
    return eng.verify_batch_grouped_packed(2, 0, s["pk"], s["sg"], s["idx"], s["data"], s["off"])


def run_batch(eng, s):
    return eng.verify_batch_packed(2, 0, s["pk"], s["sg"], s["data_items"], s["off_items"])


def held_by_fresh_context(B, fn, s):
    """device memory a fresh context holds after one call of fn (bytes)"""
    import torch
    torch.cuda.synchronize()
    free0, _ = torch.cuda.mem_get_info(0)
    e = B.Engine([0])
    fn(e, s)
    free1, _ = torch.cuda.mem_get_info(0)
    e.close()
    return int(free0 - free1)


def measure(B, s, reps, bad):
    """timing on a context of its own, closed before the arena of each call is read on a fresh one"""
    out = {}
    res = {}
    eng = B.Engine([0])
    for name, fn in (("grouped", run_grouped), ("verify_batch", run_batch)):
        res[name] = fn(eng, s)  # warm-up
        out[name] = dict(wall_ms=[])
    for _ in range(reps):
        for name, fn in (("grouped", run_grouped), ("verify_batch", run_batch)):
            t0 = time.perf_counter()
            st = fn(eng, s)
            out[name]["wall_ms"].append((time.perf_counter() - t0) * 1e3)
            out[name]["stage_ms"] = eng.last_stage_ms()
            out[name]["kernel_ms"] = {k: [round(ms, 3), c] for k, (ms, c) in eng.last_kernel_ms().items()}
            assert st.tolist() == res[name].tolist()
    eng.close()
    assert res["grouped"].tobytes() == res["verify_batch"].tobytes()
    assert np.flatnonzero(res["grouped"]).tolist() == bad
    for name, fn in (("grouped", run_grouped), ("verify_batch", run_batch)):
        o = out[name]
        o["wall_ms_median"] = float(np.median(o["wall_ms"]))
        o["sigs_per_s"] = N / (o["wall_ms_median"] / 1e3)
        o["arena_bytes"] = held_by_fresh_context(B, fn, s)
    out["speedup"] = out["verify_batch"]["wall_ms_median"] / out["grouped"]["wall_ms_median"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--shapes", default="A,B,C,D,E")
    ap.add_argument("--label", default="", help="recorded in the JSON (e.g. the library variant BLSGPU_LIB points at)")
    a = ap.parse_args()
    import blsful_b200 as B
    os.makedirs(a.out, exist_ok=True)
    eng = B.Engine([0])
    rnd = random.Random(20261020)
    res = {"info": device_info(), "impl": "Bls12381G2Impl", "scheme": "Basic", "format": "Modern", "rlc_bits": 64, "items": N,
           "label": a.label, "shapes": {}}
    qs = {"A": 1, "B": 1000, "C": N // 2, "D": N}
    wanted = a.shapes.split(",")
    for name in ("A", "B", "C", "D", "E"):
        if name not in wanted:
            continue
        if name == "E":
            s = make_shape(eng, B, rnd, 1000)
            for nbad in (1, 1000):
                bad = sorted(random.Random(nbad).sample(range(N), nbad))
                sg = s["sg"].reshape(N, 96).copy()
                for i in bad:
                    sg[i] = s["sg"].reshape(N, 96)[(i + 1) % N]
                r = measure(B, dict(s, sg=sg.reshape(-1)), a.reps, bad)
                res["shapes"]["E%d" % nbad] = dict(q=1000, bad=nbad, **r)
                print("E%d" % nbad, json.dumps(res["shapes"]["E%d" % nbad]), flush=True)
            continue
        s = make_shape(eng, B, rnd, qs[name])
        res["shapes"][name] = dict(q=qs[name], bad=0, **measure(B, s, a.reps, []))
        print(name, json.dumps(res["shapes"][name]), flush=True)
    eng.close()
    with open(os.path.join(a.out, "verify_grouped.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

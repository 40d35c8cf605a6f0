#!/usr/bin/env python
"""bench.py - verified signatures/s of the batch verification hot path (BASELINE.json metric).

Workload (configs[1]): Bls12381G2Impl batch verify of N_SIGS distinct-message signatures (hash_to_curve + pairing),
from compressed bytes.  A "step" is one pass of blsgpu_verify_batch over one batch.  Per rank (one process per GPU,
no data-path collective, weak scaling): every rank verifies its own batch.

  value : sigs/s with the batch already resident in HBM (blsgpu_verify_batch_dev), CUDA events on the launching stream
  e2e   : sigs/s through the host-buffer C-ABI call (pinned host inputs, H2D + D2H inside the timed region)
  roofline : INT32 multiply-accumulate (IMAD.WIDE) rate of the dominant kernel against the rate measured on this
             GPU by blsgpu_imad_peak.  The path is integer-multiply bound: the largest HBM stream (the Miller line
             records, 39 KB per signature written once and read once) is ~80 GB per 1M batch = 12 ms at 6.5 TB/s,
             against ~1 s of arithmetic.
  cpu_baseline : the CPU oracle restating the reference's per-signature core_verify, timed on a bounded sample

`--impl reference` times the reference's CPU path (oracle restatement: blsful itself needs cargo + un-vendored crates).
`--dump-outputs DIR` writes the status vectors of the last timed step of each leg as DIR/<name>.npy (float32); the inputs
are seeded, so two builds run with the same arguments can be compared output for output.  The benchmark batch is all
valid, so those vectors are all zero; planted_status.npy adds the statuses of the same device call, untimed, on a copy of
the batch with a seeded set of planted rejections (see plant_rejections).
"""
import argparse
import gc
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "agora-blsful_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)
sys.dont_write_bytecode = True  # the benchmark leaves the source tree as it found it

import numpy as np

METRIC = "verified sigs/sec, 1M-batch G2Impl"
UNIT = "sigs/s"
# algorithmic work per unit (SURVEY.md 8d / BASELINE.md 4): Fp-mul = 300 32x32->64 multiply-accumulates
MAC_PER_FPMUL = 300
FPMUL_PER_SIG = 14400
FPMUL_PER_STAGE = {  # per signature, from compressed bytes (SURVEY.md 8d breakdown)
    "decode_pk": 1510, "decode_sig": 2200, "hash_to_curve": 5300, "miller": 790 + 4450, "scale_sig": 120,
    "reduce": 10, "final": 0, "bisect": 0,
}
# the same breakdown per kernel launch (SURVEY.md 8a-a8 / 8d: Fp sqrt chain 460 + G1 subgroup check ~1,000 + glue;
# Fp2 sqrt ~1,000 + G2 subgroup check ~1,200; hash: 2 SSWU 2,020 + isogenies/add 140 + hash_to_field 8 | cofactor 2,630 |
# normalise 480; Miller: r_i*pk_i 790 | line steps 63*25 + 5*41 | line multiplications 68*39)
FPMUL_PER_KERNEL = {
    "k_decode_pk": 510, "k_subgroup_check_pk": 1000, "k_decode_sig": 1000, "k_subgroup_check_sig": 1200,
    "k_hash": 2168, "k_clear_cofactor": 2630, "k_to_affine_batch": 480,
    "k_m6_prep": 790, "k_m6_lines": 1780, "k_m6_accum": 2670,
}


def synth_batch(eng, n, seed, impl=2, scheme=0):
    """Deterministic synthetic triples: 31-byte random scalars (non-zero, < r), distinct 32-byte messages; signatures are
    produced once by the engine's synthetic-data helper (signing is not part of the measured path)."""
    import blsful_b200 as B
    rng = np.random.Generator(np.random.Philox(key=seed))
    scal = np.zeros((n, 32), dtype=np.uint8)
    scal[:, 1:] = rng.integers(0, 256, size=(n, 31), dtype=np.uint8)
    scal[:, 31] |= 1
    msgs = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    msgs[:, :8] = np.arange(n, dtype=np.uint64).view(np.uint8).reshape(n, 8)  # distinct by construction
    off = (np.arange(n + 1, dtype=np.uint64) * 32)
    pks = np.empty(n * B.pk_len(impl), dtype=np.uint8)
    sigs = np.empty(n * B.sig_len(impl), dtype=np.uint8)
    chunk = 1 << 18
    for lo in range(0, n, chunk):
        hi = min(n, lo + chunk)
        o = off[lo:hi + 1] - off[lo]
        p, s = eng.testdata_sign(impl, scheme, scal[lo:hi].reshape(-1), msgs[lo:hi].reshape(-1), np.ascontiguousarray(o))
        pks[lo * B.pk_len(impl):hi * B.pk_len(impl)] = p
        sigs[lo * B.sig_len(impl):hi * B.sig_len(impl)] = s
    return pks, sigs, msgs.reshape(-1), off


class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
            nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
            nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake",
        }
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.5)  # a few samples per second are enough for a median; NVML queries contend with kernel launches

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unsampled"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def cpu_baseline(batch, sample):
    """The reference's per-signature path (Signature::verify -> core_verify: decode + subgroup checks, hash_to_curve, 2 Miller
    loops, 1 final exponentiation per signature) run by the C oracle on the first `sample` signatures of the benchmark batch."""
    from oracle import cpu_verify
    pks, sigs, msgs, off = batch
    k = min(sample, off.size - 1)
    return cpu_verify.time_verify_sample((pks[:48 * k], sigs[:96 * k], msgs[:int(off[k])], off[:k + 1]))


def run_reference(args, rank, world):
    if rank != 0:
        return
    from oracle import cpu_verify
    res = cpu_verify.reference_arm(n_per_step=args.ref_sample, steps=args.steps, warmup=args.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u32 limbs (381-bit modular integers)", "data": "synthetic",
        "config": {"workload": "Bls12381G2Impl Basic Signature::verify over distinct (pk, 32-byte msg, sig) triples from compressed bytes "
                               "(the per-item work of the 1M batch; configs[0] shape), per-signature reference CPU path",
                   "sample_sigs_per_step": res["n_per_step"]},
        "cpu_baseline": {"value": res["value"], "unit": UNIT, "cores": res["cores"], "kind": res["kind"], "sample": res["sample"]},
        "e2e": {"value": res["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def _ms(fn, reps=1):
    """Wall time of a synchronous host call (every C-ABI entry point returns after its results are in host memory)."""
    best = None
    for _ in range(reps):
        t0 = time.perf_counter()
        r = fn()
        dt = (time.perf_counter() - t0) * 1e3
        best = dt if best is None or dt < best else best
    return r, best


def other_configs(eng, B, batch, peak_mac, quorums):
    """The other BASELINE.json configs and the failure path, once each, through the host-buffer C-ABI calls (H2D/D2H inside
    the timed call).  Every result is checked by construction (valid data verifies, planted failures are found exactly)."""
    pks, sigs, msgs, off = batch
    n = off.size - 1
    out = {}

    def frac(fp_mul_per_item, items, ms):
        return items * fp_mul_per_item * MAC_PER_FPMUL / (ms * 1e-3) / peak_mac

    # cfg 1: 1,024 distinct triples (latency of a small batch)
    m = min(1024, n)
    sub = (pks[:48 * m], sigs[:96 * m], msgs[:int(off[m])], off[:m + 1])
    eng.verify_batch_packed(2, 0, *sub)
    st, ms = _ms(lambda: eng.verify_batch_packed(2, 0, *sub), 3)
    assert int(st.max()) == 0
    out["cfg1_verify_1024_triples"] = {"ms": ms, "items_per_s": m / (ms * 1e-3), "note": "latency-bound: 1,024 items do not fill 148 SMs"}
    # cfg 2 failure path: 1 and 1,000 corrupted signatures (exact bad set through bisection)
    rng = np.random.default_rng(1)
    st, ms0 = _ms(lambda: eng.verify_batch_packed(2, 0, pks, sigs, msgs, off))
    assert int(st.max()) == 0
    out["cfg2_all_valid_host_call"] = {"ms": ms0, "items_per_s": n / (ms0 * 1e-3)}
    for nbad in (1, 1000):
        if nbad >= n:
            continue
        bad = np.sort(rng.choice(n, nbad, replace=False))
        s2 = sigs.copy().reshape(n, 96)
        s2[bad] = s2[(bad + 1) % n]
        st, ms = _ms(lambda: eng.verify_batch_packed(2, 0, pks, s2.reshape(-1), msgs, off))
        assert np.array_equal(np.nonzero(st)[0], bad) and set(st[bad].tolist()) == {1}
        out[f"cfg2_{nbad}_bad"] = {"ms": ms, "items_per_s": n / (ms * 1e-3), "vs_all_valid": ms / ms0}
    # cfg 2 with 128-bit random-linear-combination scalars
    eng.set_rlc_bits(128)
    st, ms = _ms(lambda: eng.verify_batch_packed(2, 0, pks, sigs, msgs, off))
    eng.set_rlc_bits(64)
    assert int(st.max()) == 0
    out["cfg2_rlc_128bit"] = {"ms": ms, "items_per_s": n / (ms * 1e-3), "vs_64bit": ms / ms0}
    # cfg 4: AggregateSignature::verify over 100k distinct messages
    m4 = min(100_000, n)
    agg = eng.sum_points(2, sigs[:m4 * 96])
    msgs_list = [msgs[int(off[i]):int(off[i + 1])].tobytes() for i in range(m4)]
    eng.aggregate_verify(2, 0, pks[:m4 * 48], msgs_list, agg)
    _, ms = _ms(lambda: eng.aggregate_verify(2, 0, pks[:m4 * 48], msgs_list, agg))
    out["cfg4_aggregate_verify_100k"] = {"ms": ms, "items_per_s": m4 / (ms * 1e-3), "frac": frac(11300, m4, ms),
                                         "note": "includes packing 100k Python byte strings on the host"}
    # Bls12381G1Impl batch verify and cfg 3 (same-message aggregation of n signers, PoP scheme), both impls
    scal = np.zeros((n, 32), dtype=np.uint8)
    scal[:, 8:] = rng.integers(0, 256, size=(n, 24), dtype=np.uint8)
    scal[:, 31] |= 1
    one_msg = np.frombuffer(b"one message for every signer....", dtype=np.uint8)
    chunk = 1 << 18
    for impl_id, pkg, sgg in ((2, 1, 2), (1, 2, 1)):
        pl, sl = B.pk_len(impl_id), B.sig_len(impl_id)
        pk3, sg3 = np.empty(n * pl, dtype=np.uint8), np.empty(n * sl, dtype=np.uint8)
        for lo in range(0, n, chunk):
            hi = min(n, lo + chunk)
            o = np.arange(hi - lo + 1, dtype=np.uint64) * 32
            p, g = eng.testdata_sign(impl_id, 2, scal[lo:hi].reshape(-1), np.tile(one_msg, hi - lo), o)
            pk3[lo * pl:hi * pl], sg3[lo * sl:hi * sl] = p, g
        apk, t1 = _ms(lambda: eng.sum_points(pkg, pk3))
        asg, t2 = _ms(lambda: eng.sum_points(sgg, sg3))
        st, t3 = _ms(lambda: eng.verify_batch(impl_id, 2, [apk], [asg], [one_msg.tobytes()]))
        assert st.tolist() == [0]
        name = "G2Impl" if impl_id == 2 else "G1Impl"
        out[f"cfg3_aggregate_{n}_signers_{name}"] = {"ms": t1 + t2 + t3, "sum_pk_ms": t1, "sum_sig_ms": t2, "verify_ms": t3,
                                                      "items_per_s": n / ((t1 + t2 + t3) * 1e-3), "frac": frac(3750, n, t1 + t2 + t3)}
        if impl_id == 1:
            # G1Impl distinct-message batch verify (signatures in G1, keys in G2)
            p1, s1, m1, o1 = synth_batch(eng, n, seed=4242, impl=1)
            eng.verify_batch_packed(1, 0, p1, s1, m1, o1)
            st, ms = _ms(lambda: eng.verify_batch_packed(1, 0, p1, s1, m1, o1))
            assert int(st.max()) == 0
            out["G1Impl_batch_verify"] = {"ms": ms, "items_per_s": n / (ms * 1e-3), "n": n}
    # cfg 5: verify_secure / aggregate_secure over quorums of 400 members, Modern and Legacy
    q, mem = quorums, 400
    tot = q * mem
    sc5 = np.zeros((tot, 32), dtype=np.uint8)
    sc5[:, 8:] = rng.integers(0, 256, size=(tot, 24), dtype=np.uint8)
    sc5[:, 31] |= 1
    qm = rng.integers(0, 256, size=(q, 32), dtype=np.uint8)
    qm[:, :8] = np.arange(q, dtype=np.uint64).view(np.uint8).reshape(q, 8)
    pk5, sg5 = np.empty(tot * 48, dtype=np.uint8), np.empty(tot * 96, dtype=np.uint8)
    for lo in range(0, tot, chunk):
        hi = min(tot, lo + chunk)
        o = np.arange(hi - lo + 1, dtype=np.uint64) * 32
        p, g = eng.testdata_sign(2, 0, sc5[lo:hi].reshape(-1), np.ascontiguousarray(qm[np.arange(lo, hi) // mem]).reshape(-1), o)
        pk5[lo * 48:hi * 48], sg5[lo * 96:hi * 96] = p, g
    koff = np.arange(q + 1, dtype=np.uint64) * mem
    qoff = np.arange(q + 1, dtype=np.uint64) * 32
    for fmt, fname in ((1, "modern"), (0, "legacy")):
        if fmt == 0:
            pk5 = eng.recode_points_packed(1, pk5, 1, 0)
            sg5 = eng.recode_points_packed(2, sg5, 1, 0)
        (stq, aggs), ta = _ms(lambda: eng.aggregate_secure_batch_packed(2, koff, pk5, sg5, fmt))
        assert int(stq.max()) == 0
        st, tv = _ms(lambda: eng.verify_secure_batch_packed(2, 0, koff, pk5, aggs, qm.reshape(-1), qoff, fmt))
        assert int(st.max()) == 0
        swapped = aggs.copy().reshape(q, 96)
        if q > 4:
            swapped[[3, 4]] = swapped[[4, 3]]
            st = eng.verify_secure_batch_packed(2, 0, koff, pk5, swapped.reshape(-1), qm.reshape(-1), qoff, fmt)
            assert np.nonzero(st)[0].tolist() == [3, 4]
        out[f"cfg5_verify_secure_{q}x{mem}_{fname}"] = {"ms": tv, "members_per_s": tot / (tv * 1e-3), "quorums_per_s": q / (tv * 1e-3),
                                                        "frac": frac(2400, tot, tv)}
        out[f"cfg5_aggregate_secure_{q}x{mem}_{fname}"] = {"ms": ta, "members_per_s": tot / (ta * 1e-3)}
    return out


_RESULT_FD = None


def _claim_stdout():
    """stdout carries exactly ONE JSON line: anything libraries print there (NCCL's version banner under NCCL_DEBUG, for
    one) is sent to stderr instead; emit() writes the result to the real stdout."""
    global _RESULT_FD
    sys.stdout.flush()
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)


def emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_RESULT_FD, data)


DUMP_BYTES = 64 << 20


def dump_outputs(dirname, arrays):
    """Writes each array as dirname/<name>.npy in float32.  If they would take more than DUMP_BYTES together, every array
    is cut to the same fixed, seeded sample of positions, written beside it as <name>_index.npy (float64)."""
    os.makedirs(dirname, exist_ok=True)
    total = sum(a.size for a in arrays.values()) * 4
    for i, (name, a) in enumerate(arrays.items()):
        a = np.asarray(a).reshape(-1)
        if total > DUMP_BYTES:
            k = min(a.size, DUMP_BYTES // (len(arrays) * 12))   # 4 B per value + 8 B per index
            idx = np.sort(np.random.default_rng(i).choice(a.size, k, replace=False))
            np.save(os.path.join(dirname, f"{name}_index.npy"), idx.astype(np.float64))
            a = a[idx]
        np.save(os.path.join(dirname, f"{name}.npy"), a.astype(np.float32))


def plant_rejections(pks, sigs, n, seed=7):
    """A copy of a G2Impl batch (48 B keys, 96 B signatures) with k = min(64, n // 8) items of each kind the verifier must
    reject, at fixed, seeded positions, and the statuses it must return: another item's signature (1), the identity
    signature (2), the identity public key (3), an undecodable public key (4).  Everything else keeps status 0."""
    k = min(64, n // 8)
    pos = np.random.default_rng(seed).choice(n, 4 * k, replace=False).reshape(4, k)
    p, s = pks.reshape(n, 48).copy(), sigs.reshape(n, 96).copy()
    s[pos[0]] = sigs.reshape(n, 96)[(pos[0] + 1) % n]
    s[pos[1]] = 0
    s[pos[1], 0] = 0xC0
    p[pos[2]] = 0
    p[pos[2], 0] = 0xC0
    p[pos[3]] = 0
    want = np.zeros(n, dtype=np.uint8)
    for status, idx in enumerate(pos, 1):
        want[idx] = status
    return p.reshape(-1), s.reshape(-1), want


def _positive(s):
    v = int(s)
    if v < 1:
        raise argparse.ArgumentTypeError("must be at least 1")
    return v


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=_positive, default=3, help="timed steps of every leg")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--n", type=int, default=int(os.environ.get("BLSGPU_BENCH_N", 1_000_000)), help="signatures per batch per GPU")
    ap.add_argument("--ref-sample", type=int, default=0, help="signatures per step for --impl reference (0 = 1,024: configs[0])")
    ap.add_argument("--cpu-sample", type=int, default=0, help="signatures for the cpu_baseline leg (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the other BASELINE.json configs (cfg 1, 3, 4, 5, failure path)")
    ap.add_argument("--quorums", type=int, default=int(os.environ.get("BLSGPU_BENCH_QUORUMS", 10_000)), help="cfg 5 quorums of 400 members")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the status vectors of the last timed step of each leg, and of one untimed call on the batch "
                         "with planted rejections, as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    _claim_stdout()

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))

    if args.impl == "reference":
        if args.dump_outputs:
            raise SystemExit("bench.py: --dump-outputs applies to the engine (--impl engine)")
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import blsful_b200 as B

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the engine has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    eng = B.Engine([local_rank])
    stream = torch.cuda.Stream(device=dev)
    eng.set_stream(stream.cuda_stream)
    impl, scheme, n = B.Bls12381G2Impl, B.SignatureSchemes.Basic, args.n

    peak_mac = eng.imad_peak()
    lo, hi = B.shard_range(world * n, rank, world)  # weak scaling: the job is world*n signatures, rank r owns [lo, hi)
    assert hi - lo == n
    pks, sigs, msgs, off = synth_batch(eng, n, seed=1000 + rank)

    # pinned host copies (e2e leg) and device-resident copies (value leg)
    def pinned(a):
        t = torch.from_numpy(a).pin_memory()
        return t
    h_pk, h_sig, h_msg, h_off = pinned(pks), pinned(sigs), pinned(msgs), pinned(off.view(np.int64))
    d_pk, d_sig, d_msg, d_off = (t.to(dev) for t in (h_pk, h_sig, h_msg, h_off))
    d_status = torch.empty(n, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()

    def step_dev():
        eng.verify_batch_dev(impl, scheme, n, d_pk.data_ptr(), d_sig.data_ptr(), d_msg.data_ptr(), d_off.data_ptr(), d_status.data_ptr())

    np_pk, np_sig, np_msg, np_off = h_pk.numpy(), h_sig.numpy(), h_msg.numpy(), h_off.numpy().view(np.uint64)

    host_ms, host_dev_ms = [], []
    last = {}  # the statuses each leg returned in its latest step (--dump-outputs)

    def step_host():
        t0 = time.perf_counter()
        st = eng.verify_batch_packed(impl, scheme, np_pk, np_sig, np_msg, np_off)
        host_ms.append((time.perf_counter() - t0) * 1e3)
        host_dev_ms.append(sum(eng.last_stage_ms().values()))
        last["e2e_status"] = st
        return st

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        gc.collect()
        gc.disable()  # a collection inside the host-buffer call showed up as a 25 ms outlier in one of three steps
        try:
            return _timed(fn, steps)
        finally:
            gc.enable()

    def _timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            fn()
        e1.record(stream)
        e1.synchronize()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    for _ in range(args.warmup):
        step_dev()
    assert int(d_status.max().item()) == 0, "synthetic batch must verify"
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = eng.launch_count()
    ms_total = timed(step_dev, args.steps)
    launches = eng.launch_count() - launches0
    stages = eng.last_stage_ms()
    kernels = eng.last_kernel_ms()
    sampler.stop_flag = True
    sampler.join(timeout=2)
    last["verify_status"] = d_status.cpu().numpy()
    assert int(last["verify_status"].max()) == 0

    # e2e through the host-buffer call
    for _ in range(max(1, args.warmup)):  # the same W warm-up calls as the device leg (the first calls grow the arena)
        st = step_host()
    assert int(st.max()) == 0
    e2e_steps = args.steps
    ms_e2e = timed(step_host, e2e_steps)

    value = world * n * args.steps / (ms_total * 1e-3)
    e2e_value = world * n * e2e_steps / (ms_e2e * 1e-3)

    # roofline of the dominant kernel: every hot kernel has its own CUDA-event pair on the stream it is launched on
    # (blsgpu_last_kernel_ms, last timed step); dominant = the longest.  Algorithmic MACs per launch / launch duration.
    per_kernel = {}
    for k, (ms, cnt) in kernels.items():
        if cnt == 0 or ms <= 0:
            continue
        macs = n * FPMUL_PER_KERNEL[k] * MAC_PER_FPMUL / cnt          # per launch
        per_kernel[k] = {"ms_per_launch": ms / cnt, "launches_per_step": cnt, "fp_mul_per_sig": FPMUL_PER_KERNEL[k],
                         "frac": macs / (ms / cnt * 1e-3) / peak_mac}
    dom = max(per_kernel, key=lambda k: per_kernel[k]["ms_per_launch"] * per_kernel[k]["launches_per_step"])
    achieved = per_kernel[dom]["frac"] * peak_mac / 1e9
    whole = n * FPMUL_PER_SIG * MAC_PER_FPMUL / ((ms_total / args.steps) * 1e-3) / 1e9
    per_stage = {k: {"ms": v, "fp_mul_per_sig": FPMUL_PER_STAGE[k],
                     "frac": (n * FPMUL_PER_STAGE[k] * MAC_PER_FPMUL / (v * 1e-3) / peak_mac) if v > 0 else None}
                 for k, v in stages.items()}
    traffic = None
    try:  # dram bytes per launch of the dominant kernel from the committed ncu capture of this round (profiles/)
        tp = os.path.join(ROOT, "profiles", "traffic_r2.json")
        tr = json.load(open(tp if os.path.exists(tp) else os.path.join(ROOT, "profiles", "traffic_r1.json")))
        traffic = tr.get(dom, {}).get("dram_bytes_per_sig", None)
        traffic = traffic * n / per_kernel[dom]["launches_per_step"] if traffic is not None else None
    except Exception:
        pass
    roofline = {
        "bound": "int32_imad (not hbm, not tensor: see DESIGN.md section 6)", "kernel": dom, "achieved": achieved,
        "peak": peak_mac / 1e9, "unit": "GMAC/s", "frac": achieved / (peak_mac / 1e9), "traffic": traffic,
        "whole_step": {"achieved": whole, "frac": whole / (peak_mac / 1e9), "fp_mul_per_sig": FPMUL_PER_SIG},
        "peak_source": "measured live by blsgpu_imad_peak (8 independent IMAD.WIDE.U32 chains per thread with changing "
                       "operands on all SMs); MEASURED_PEAKS.json holds no INT32 figure; ncu counterpart: "
                       "sm__pipe_fmaheavy_cycles_active",
        "algorithmic_unit": "1 Fp-mul = 300 32x32->64 MACs (SURVEY.md 8d); the kernels execute 357 (Karatsuba, 28-bit radix)",
        "kernels": per_kernel, "stages": per_stage,
    }

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u32 limbs (381-bit modular integers)", "data": "synthetic",
        "config": {"workload": f"Bls12381G2Impl Basic batch verify, {n} distinct 32-byte messages per GPU, compressed inputs "
                               "(48 B pk + 96 B sig), hash_to_curve + pairing, all valid",
                   "sigs_per_gpu": n, "l2": "inputs (176 B/sig) and the 39 KB/sig Miller line records exceed L2 at 1M: everything streams through HBM",
                   "miller_loops_per_s_per_gpu": (n / (stages["miller"] * 1e-3)) if stages.get("miller") else None,
                   "miller_loops_note": "n Miller loops / device time of the Miller stage (prep + lines + accumulator kernels)"},
        "roofline": roofline, "clocks": sampler.summary(),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(n * 176 + (n + 1) * 8), "d2h_bytes_per_step": int(n),
                "host_call_ms": [round(x, 1) for x in host_ms[-e2e_steps:]],
                "host_call_device_ms": [round(x, 1) for x in host_dev_ms[-e2e_steps:]]},
        "gpu_launches": int(launches),
    }
    # strong scaling: ONE batch of n signatures cut over the ranks; every rank folds its slice into one partial product of
    # Miller values + one partial sum, the 672-byte partial results are exchanged (NCCL all_gather), every rank runs the single
    # Miller loop + final exponentiation of the whole batch and finishes its slice (SURVEY.md 8e; host buffers in and out)
    def all_gather_parts(part):
        mine = torch.tensor(list(part[0] + part[1]), dtype=torch.uint8, device=dev)
        outs = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(outs, mine)
        return [(bytes(o[:576].tolist()), bytes(o[576:].tolist())) for o in outs]

    if rank == 0 or world == 1:
        s_pk, s_sig, s_msg, s_off = np_pk, np_sig, np_msg, np_off
    else:  # the SAME batch on every rank (rank 0's): each rank verifies its slice of it
        s_pk, s_sig, s_msg, s_off = synth_batch(eng, n, seed=1000)

    def step_strong():
        r = B.verify_batch_folded(eng, impl, scheme, s_pk, s_sig, s_msg, s_off, rank, world, all_gather_parts)
        last["strong_status"] = r[1]
        return r

    lo_s, st = step_strong()
    assert int(st.max()) == 0
    ms_strong = timed(step_strong, e2e_steps)
    line["strong_scaling"] = {"batch": n, "n_gpus": world, "ms_per_batch": ms_strong / e2e_steps, "value": n * e2e_steps / (ms_strong * 1e-3),
                              "unit": UNIT, "exchange_bytes_per_rank": 672,
                              "what": "ONE batch cut over the ranks: per-rank partial Fp12 + partial sum, all_gather, single final exponentiation"}
    if rank == 0 and args.dump_outputs:
        # the timed batch is all valid, so its statuses cannot tell a correct build from one that accepts everything:
        # the same device call, after the timed legs, on a copy with planted rejections
        p_pk, p_sig, want = plant_rejections(pks, sigs, n)
        d_ppk, d_psig = torch.from_numpy(p_pk).to(dev), torch.from_numpy(p_sig).to(dev)
        d_pstatus = torch.empty(n, dtype=torch.uint8, device=dev)
        torch.cuda.synchronize()
        eng.verify_batch_dev(impl, scheme, n, d_ppk.data_ptr(), d_psig.data_ptr(), d_msg.data_ptr(), d_off.data_ptr(), d_pstatus.data_ptr())
        stream.synchronize()
        last["planted_status"] = d_pstatus.cpu().numpy()
        dump_outputs(args.dump_outputs, last)
        assert np.array_equal(last["planted_status"], want), "the planted rejections must be found exactly"
    if rank == 0 and world == 1 and not args.no_configs:
        line["configs"] = other_configs(eng, B, (pks, sigs, msgs, off), peak_mac, args.quorums)
    if rank == 0 and not args.no_cpu_baseline and world == 1:
        line["cpu_baseline"] = cpu_baseline((pks, sigs, msgs, off), args.cpu_sample or 256 * (os.cpu_count() or 1))
    if rank == 0:
        emit(line)
    eng.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

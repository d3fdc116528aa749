#!/usr/bin/env python3
"""bench.py -- BLS12-381 G1 scalar-muls/sec through the Pippenger MSM hot path (BASELINE.json configs[1]).

  python bench.py --gpus N --steps K --warmup W            # our arm (sm_100a kernels via the C ABI)
  python bench.py --impl reference --gpus N --steps K ...  # CPU arm: the reference's algorithm (oracle port)

A "step" is one MSM over one resident batch of 2^20 (scalar, point) pairs per GPU (weak scaling: rank r
owns pairs [r*n, (r+1)*n) of an N*n-pair MSM; partial sums are exchanged with ONE NCCL all-gather of
96-byte affine points and added on every rank).  `value` = pairs / device time with inputs resident in
HBM; `e2e` = the same through b2k_bls12381_g1_msm with pinned HOST buffers (H2D of scalars+points and
D2H of the result inside the timed region).  Results are checked against the oracle every run
(sum s_i*(a_i*G) == (sum s_i a_i mod r)*G).
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# several contexts per rank, each with device-side waits on flags other streams / ranks set: one hardware queue per stream
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

METRIC = "bls12381_g1_scalar_muls_per_sec"
UNIT = "scalar-muls/s"
LOG_N = int(os.environ.get("B2K_BENCH_LOGN", "20"))


# ------------------------------------------------------------------------------------------------
def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index = index
        self.rows = []
        self.stop_flag = False
        self.proc = None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append(line.strip())
                if self.stop_flag:
                    break
        except Exception:
            pass

    def finish(self):
        self.stop_flag = True
        if self.proc:
            try:
                self.proc.terminate()
            except Exception:
                pass
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = max(mx, float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        med = sm[len(sm) // 2] if sm else None
        return {"sm_mhz": med, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
def best_cpu_threads() -> int:
    """Threads of the CPU arm: FIXED rule, printed in the JSON -- min(32, logical CPUs) (B2K_REF_THREADS overrides).
    On the 128-logical-CPU GPU boxes 32 threads measured fastest for this memory-light, multiply-bound loop in round 1
    (64 / 128 lose to SMT sharing and the container's CPU quota); a per-run calibration made the baseline itself vary 2x."""
    v = os.environ.get("B2K_REF_THREADS")
    if v and v.isdigit() and int(v) > 0:
        return int(v)
    return max(1, min(32, os.cpu_count() or 1))


def cpu_sample(n_sample: int, threads: int, seed_start: int = 0):
    """n_sample pairs of the C2 workload: points a_i * G made by the CPU port itself (operand form, no per-point Python)"""
    from kyber_b200 import workload as wl
    from oracle import cpu_ref
    lib = cpu_ref.load()
    s = wl.prng_scalars("b2k/c2", n_sample, wl.R_BLS12381, seed_start)
    a = wl.prng_scalars("b2k/c2-a", n_sample, wl.R_BLS12381, seed_start)
    pts = cpu_ref.g1_mul_batch_affine(lib, wl.scalars_to_bytes(a), wl.G1_BLS12381_AFFINE * n_sample, os.cpu_count() or threads)
    return lib, s, a, wl.scalars_to_bytes(s), pts


def cpu_reference_run(n_sample: int, threads: int, seed_start: int = 0, with_pippenger: bool = True):
    """Time the oracle's restatement of the reference path (N x Point.Mul + Add, share/poly.go:461-473)
    and, separately, a CPU Pippenger, on a bounded sample of the same workload."""
    from kyber_b200 import workload as wl
    from oracle import cpu_ref
    from oracle import bls12381 as o
    lib, s, a, sb, pts = cpu_sample(n_sample, threads, seed_start)
    t0 = time.perf_counter()
    out = cpu_ref.g1_msm_muladd(lib, sb, pts, threads)
    t_muladd = time.perf_counter() - t0
    expect = o.g1_compress(o.g1_mul(wl.dot_mod(s, a, o.R)))
    assert out == expect, "CPU reference arm produced a wrong MSM"
    res = {"value": n_sample / t_muladd, "unit": UNIT, "cores": threads, "kind": "port",
           "sample": f"{n_sample} pairs of the 2^20 workload: Mul+Add loop (the reference's algorithm, "
                     f"share/poly.go:461-473) on {threads} threads, {t_muladd:.2f} s; oracle/cpu_ref.c "
                     "(C restatement, NOT the Go reference: no Go toolchain on this image)",
           "seconds": t_muladd}
    if with_pippenger:
        t0 = time.perf_counter()
        out2 = cpu_ref.g1_msm_pippenger(lib, sb, pts, threads)
        t_pip = time.perf_counter() - t0
        assert out2 == expect
        res["pippenger_value"] = n_sample / t_pip
        res["pippenger_note"] = ("same sample through a multi-threaded CPU Pippenger (a stronger baseline than the "
                                 "reference, which has no MSM)")
    return res


def cpu_pairing_run(n_sample: int, threads: int):
    """CPU baseline for pairings/s: n_sample 2-pair checks (ValidatePairing, kilic/suite.go:57-68) on all threads."""
    from oracle import cpu_ref
    from oracle import bls12381 as o
    lib = cpu_ref.load()
    x, y = 0x1234567, 0x89abcdef
    a1 = o.g1_to_affine_bytes(o.g1_mul(x)) * n_sample
    a2 = o.g2_to_affine_bytes(o.g2_mul(y)) * n_sample
    b1 = o.g1_to_affine_bytes(o.g1_mul(x * y)) * n_sample
    b2 = o.g2_to_affine_bytes(o.G2) * n_sample
    t0 = time.perf_counter()
    ok = cpu_ref.pairing_check(lib, a1, a2, b1, b2, threads)
    dt = time.perf_counter() - t0
    assert set(ok) == {1}
    return {"value": 2 * n_sample / dt, "unit": "pairings/s", "cores": threads, "kind": "port",
            "sample": f"{n_sample} ValidatePairing checks (2 pairings each) on {threads} threads, {dt:.2f} s; "
                      "oracle/cpu_ref.c (C restatement, NOT the Go reference)"}


def gpu_pairing_run(eng, torch, dev, n: int, steps: int):
    """pairings/s on the GPU: n independent ValidatePairing checks per step (BASELINE configs[2] mode A's
    pairing stage), operands resident in HBM; verified (all ones, one corrupted element zero)."""
    from oracle import bls12381 as o
    x, y = 0x1234567, 0x89abcdef
    a1 = torch.frombuffer(bytearray(o.g1_to_affine_bytes(o.g1_mul(x)) * n), dtype=torch.uint8).to(dev)
    a2 = torch.frombuffer(bytearray(o.g2_to_affine_bytes(o.g2_mul(y)) * n), dtype=torch.uint8).to(dev)
    good = o.g1_to_affine_bytes(o.g1_mul(x * y))
    hb1 = bytearray(good * n)
    hb1[96 * 7:96 * 8] = o.g1_to_affine_bytes(o.g1_mul(x * y + 1))      # one wrong element
    b1 = torch.frombuffer(hb1, dtype=torch.uint8).to(dev)
    b2 = torch.frombuffer(bytearray(o.g2_to_affine_bytes(o.G2) * n), dtype=torch.uint8).to(dev)
    ok = torch.zeros(n, dtype=torch.uint8, device=dev)

    def step():
        eng._check(eng.lib.b2k_bls12381_pairing_check_dev(eng.h, n, a1.data_ptr(), a2.data_ptr(), b1.data_ptr(),
                                                          b2.data_ptr(), ok.data_ptr()))
    step(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    res = ok.cpu()
    assert int(res.sum()) == n - 1 and int(res[7]) == 0, "pairing check results wrong"
    # small batches (the one-at-a-time interface methods): the warp-cooperative kernel, one warp per check
    small = {}
    for m in (1, 1024):
        ok.zero_()
        def small_step():
            eng._check(eng.lib.b2k_bls12381_pairing_check_dev(eng.h, m, a1.data_ptr(), a2.data_ptr(), b1.data_ptr(), b2.data_ptr(), ok.data_ptr()))
        small_step(); torch.cuda.synchronize()
        e0.record()
        for _ in range(3):
            small_step()
        e1.record(); torch.cuda.synchronize()
        assert int(ok[:m].sum()) == m - (1 if m > 7 else 0), "small-batch pairing check results wrong"
        small[f"n{m}_ms"] = e0.elapsed_time(e1) / 3
    return {"value": 2 * n / (ms * 1e-3), "unit": "pairings/s", "ms_per_step": ms,
            "workload": f"{n} independent ValidatePairing checks (2-pair Miller loop + final exponentiation each)",
            "checks_per_sec": n / (ms * 1e-3), "small_batch_latency": small,
            "small_batch_note": "device time of ONE call with 1 / 1024 checks (batches <= 10240 run one check per warp, coop_pairing.cuh)"}


def gpu_mul_batch_run(eng, torch, dev, d_scal, d_pts, n: int, steps: int, scalars, a):
    """independent Point.Mul: out[i] = s_i * P_i for the step's n resident (scalar, point) pairs, no summation
    (SURVEY.md 8(d): reported beside the MSM number); a sample of the outputs is checked against the oracle."""
    from oracle import bls12381 as o
    out = torch.empty(n * 48, dtype=torch.uint8, device=dev)

    def step():
        eng.call_dev("b2k_bls12381_g1_mul_batch_dev", n, d_scal.data_ptr(), d_pts.data_ptr(), out.data_ptr())
    step(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    res = out.cpu()
    for i in (0, n // 2, n - 1):
        assert bytes(res[48 * i:48 * i + 48].tolist()) == o.g1_compress(o.g1_mul(scalars[i] * a[i] % o.R)), "mul_batch differs from the oracle"
    return {"value": n / (ms * 1e-3), "unit": "scalar-muls/s", "ms_per_step": ms,
            "workload": f"{n} independent BLS12-381 G1 Point.Mul (random 255-bit scalars, distinct points), 48-byte compressed results",
            "kernel": "k_mul_batch<Bls381G1>: endomorphism split, signed radix-16 digits over one affine table per point"}


def gpu_verify_run(eng, torch, dev, n: int, steps: int):
    """BASELINE configs[2] mode A: n independent bls.Verify (signatures on G1) per step, inputs resident in HBM:
    2 UnmarshalBinary (subgroup checks) + hash-to-G1 + ValidatePairing each; one corrupted signature must fail."""
    from oracle import bls12381 as o, h2c_bls12381 as h
    sk, msg = 0x1f2e3d4c5b6a7988, bytes(range(32))
    pk = o.g2_compress(o.g2_mul(sk))
    sig = o.g1_compress(o.g1_mul(sk, h.hash_to_g1(msg)))
    bad = o.g1_compress(o.g1_mul(sk + 1, h.hash_to_g1(msg)))
    hs = bytearray(sig * n)
    hs[48 * 5:48 * 6] = bad
    d_pk = torch.frombuffer(bytearray(pk * n), dtype=torch.uint8).to(dev)
    d_sig = torch.frombuffer(hs, dtype=torch.uint8).to(dev)
    d_msg = torch.frombuffer(bytearray(msg * n), dtype=torch.uint8).to(dev)
    d_off = torch.arange(0, 32 * (n + 1), 32, dtype=torch.int32).to(dev)
    d_dst = torch.frombuffer(bytearray(h.DST_G1), dtype=torch.uint8).to(dev)
    d_ok = torch.zeros(n, dtype=torch.uint8, device=dev)

    def step():
        eng._check(eng.lib.b2k_bls12381_verify_g1sig_dev(eng.h, n, d_pk.data_ptr(), d_msg.data_ptr(), d_off.data_ptr(),
                                                         d_dst.data_ptr(), len(h.DST_G1), d_sig.data_ptr(), d_ok.data_ptr()))
    step(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    res = d_ok.cpu()
    assert int(res.sum()) == n - 1 and int(res[5]) == 0, "verify results wrong"
    return {"value": n / (ms * 1e-3), "unit": "verifications/s", "ms_per_step": ms,
            "workload": f"{n} independent bls.Verify (sigs on G1): 2 decompress + subgroup checks, hash-to-G1, 2-pairing check"}


def section_recover_commit(eng, torch, steps: int, threads: int):
    """BASELINE configs[3] (C4): share.RecoverCommit, t = n = 1024 over bn254 G1 (share/poly.go:449-476): Lagrange + MSM on the
    device through the host C ABI (64 KiB in, 64 B out per call); result == f(0) G (oracle)."""
    from oracle import bn254 as c4
    from kyber_b200 import workload as wl
    t = 1024
    coeffs = wl.prng_scalars("b2k/c4", t, c4.ORDER)
    idx = list(range(t))
    # shares Y_i = f(i+1) G, built on the device: f(i+1) evaluated on the host (Horner over ints), one mul_batch for the points
    ev = []
    for i in idx:
        acc = 0
        for c in reversed(coeffs):
            acc = (acc * (i + 1) + c) % c4.ORDER
        ev.append(acc)
    shares = eng.bn254_g1_mul_batch(b"".join(v.to_bytes(32, "big") for v in ev), c4.g1_marshal(c4.G1) * t)
    want = c4.g1_marshal(c4.g1_mul(coeffs[0]))
    assert eng.bn254_recover_commit(idx, shares) == want, "RecoverCommit differs from f(0) G"
    t0 = time.perf_counter()
    for _ in range(steps):
        eng.bn254_recover_commit(idx, shares)
    ms = (time.perf_counter() - t0) * 1e3 / steps
    # CPU: the reference's loop = t Lagrange coefficients (O(t^2) mod.Int products) + t x (Mul + Add).  The C port has no bn254 field;
    # the EC part is quoted from the reference's own published number (95 331 ns per bn254 G1 Mul, docs/benchmark-app data.json:476)
    return {"value": 1e3 / ms, "unit": "recoveries/s", "ms_per_call": ms, "t": t,
            "workload": "share.RecoverCommit, t = n = 1024 over bn254 G1 (BASELINE.json configs[3]), host buffers in and out every call",
            "reference_published": {"ec_part_ms": 1024 * 95331e-6, "note": "1024 x bn254 G1 Point.Mul at the reference's published 95 331 ns/op "
                                    "(hardware unstated, one thread); the O(t^2) big.Int scalar part comes on top"}}


def section_bdn_aggregate(eng, torch, steps: int, threads: int):
    """BASELINE configs[2] mode B: BDN same-message aggregate over 65 536 signers (sign/bdn/bdn.go:126-181): coefficients
    (BLAKE2Xs over all public keys, host function of the library), sum (c_i+1) S_i on G1, sum (c_i+1) PK_i on G2, one bls.Verify."""
    from oracle import bls12381 as o, h2c_bls12381 as h
    from kyber_b200 import workload as wl
    n = 1 << 16
    sks = wl.prng_scalars("b2k/c3", n, o.R)
    sb = wl.scalars_to_bytes(sks)
    msg = bytes(range(32))
    hm_b = eng.bls12381_hash_to_g1([msg], h.DST_G1)
    pk_aff = eng.bls12381_g2_mul_batch_affine(sb, o.g2_to_affine_bytes(o.G2) * n)
    ones = b"".join((1).to_bytes(32, "big") for _ in range(n))
    pks = eng.bls12381_g2_mul_batch(ones, pk_aff)                         # MarshalBinary bytes the coefficients hash
    sig_aff = eng.bls12381_g1_mul_batch_affine(sb, hm_b * n)

    def once():
        cb = eng.bdn_coefficients(pks, 96, add_one=True)                  # c_i + 1, 32-byte big-endian scalars
        agg_sig = eng.bls12381_g1_msm(cb, sig_aff)
        agg_key = eng.bls12381_g2_msm(cb, pk_aff)
        ok = eng.bls12381_verify_g1sig(agg_key, [msg], h.DST_G1, agg_sig)
        return cb, agg_sig, agg_key, ok
    cb, agg_sig, agg_key, ok = once()
    coefs = [int.from_bytes(cb[32 * i:32 * i + 32], "big") for i in range(n)]
    dot = wl.dot_mod(coefs, sks, o.R)
    assert ok == b"\x01" and agg_key == o.g2_compress(o.g2_mul(dot)), "BDN aggregate differs from the oracle"
    t0 = time.perf_counter()
    for _ in range(steps):
        once()
    ms = (time.perf_counter() - t0) * 1e3 / steps
    parts = {}                                                            # where the time goes (one more pass, piece by piece)
    for name, fn in (("coefficients_host_blake2xs", lambda: eng.bdn_coefficients(pks, 96, add_one=True)),
                     ("g1_msm_signatures", lambda: eng.bls12381_g1_msm(cb, sig_aff)),
                     ("g2_msm_keys", lambda: eng.bls12381_g2_msm(cb, pk_aff)),
                     ("one_bls_verify", lambda: eng.bls12381_verify_g1sig(agg_key, [msg], h.DST_G1, agg_sig))):
        t1 = time.perf_counter()
        fn()
        parts[name] = round((time.perf_counter() - t1) * 1e3, 3)
    # CPU: the reference's loop Mul(coef, sig) + Add over the signatures (bdn.go:128-154) with the same 128-bit coefficients, bounded sample
    from oracle import cpu_ref
    lib = cpu_ref.load()
    ns = 1 << 14
    t0 = time.perf_counter()
    out = cpu_ref.g1_msm_muladd(lib, cb[:32 * ns], sig_aff[:96 * ns], threads)
    dt = time.perf_counter() - t0
    assert out == eng.bls12381_g1_msm(cb[:32 * ns], sig_aff[:96 * ns])
    return {"value": n / (ms * 1e-3), "unit": "signers/s", "ms_per_aggregate": ms, "signers": n, "parts_ms": parts,
            "parts_note": "one_bls_verify is ONE pairing check: a single thread's latency (the kernels are one check per thread), not throughput",
            "workload": "BDN aggregate of 65 536 same-message signatures (BASELINE.json configs[2] mode B): coefficients, G1 MSM of the signatures, "
                        "G2 MSM of the keys (128-bit factors c_i + 1), one bls.Verify; host buffers every call",
            "cpu_baseline": {"value": ns / dt, "unit": "signers/s", "cores": threads, "kind": "port",
                             "sample": f"AggregateSignatures only: Mul+Add loop over {ns} signatures with the same 128-bit coefficients on {threads} threads, "
                                       f"{dt:.2f} s (oracle/cpu_ref.c); the G2 key aggregation (~3x the cost per term) is not included"}}


def section_ed25519(eng, torch, steps: int):
    """BASELINE configs[0] (C1): 1024 edwards25519 Point.Mul (group/edwards25519/point.go:235-258), checked against libsodium"""
    from kyber_b200 import workload as wl
    from oracle import ed25519 as oe
    n = 1024
    L = oe.L
    sc = wl.prng_scalars("b2k/c1", n, L)
    a = wl.prng_scalars("b2k/c1-a", n, L)
    sb = b"".join(v.to_bytes(32, "little") for v in sc)
    ab = b"".join(v.to_bytes(32, "little") for v in a)
    pts = eng.ed25519_mul_batch(ab, oe.encode(oe.BASE) * n)
    out = eng.ed25519_mul_batch(sb, pts)
    cpu = None
    try:
        from nacl import bindings as nb
        t0 = time.perf_counter()
        ref = [nb.crypto_scalarmult_ed25519_noclamp(sb[32 * i:32 * i + 32], pts[32 * i:32 * i + 32]) for i in range(n)]
        dt = time.perf_counter() - t0
        assert b"".join(ref) == out, "ed25519 batch differs from libsodium"
        cpu = {"value": n / dt, "unit": "scalar-muls/s", "cores": 1, "kind": "library",
               "sample": f"{n} x libsodium crypto_scalarmult_ed25519_noclamp (PyNaCl), one thread, {dt * 1e3:.1f} ms; the reference's own "
                         "pure-Go Point.Mul is published at 349 399 ns/op (2.9e3 /s, docs/benchmark-app data.json:38)"}
    except ImportError:
        pass
    t0 = time.perf_counter()
    for _ in range(steps):
        eng.ed25519_mul_batch(sb, pts)
    ms = (time.perf_counter() - t0) * 1e3 / steps
    return {"value": n / (ms * 1e-3), "unit": "scalar-muls/s", "ms_per_batch": ms,
            "workload": "1024 edwards25519 Point.Mul (BASELINE.json configs[0]), host buffers in and out (a launch-latency-sized batch)",
            "cpu_baseline": cpu}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    threads = best_cpu_threads()
    # >= 2^16 pairs per step: >= 0.5 s of Mul+Add work at the ~1.3e5 muls/s this port reaches on 32 threads
    n_sample = int(os.environ.get("B2K_REF_SAMPLE", str(1 << 16)))
    vals, secs = [], []
    last = None
    for i in range(args.warmup + args.steps):
        last = cpu_reference_run(n_sample, threads, seed_start=i * n_sample, with_pippenger=(i == args.warmup + args.steps - 1))
        if i >= args.warmup:
            vals.append(last["value"]); secs.append(last["seconds"])
    v = sum(vals) / len(vals)
    sv = sorted(vals)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * n_sample / v,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64",
            "data": "synthetic",
            "config": {"workload": f"BLS12-381 G1 MSM, 2^{LOG_N} random (scalar,point) pairs per GPU",
                       "step": f"bounded sample of {n_sample} pairs (fresh seeds every step), {threads} threads (fixed rule: min(32, logical CPUs))"},
            "cpu_baseline": dict(last, value=v),
            "spread": {"min": sv[0], "median": sv[len(sv) // 2], "max": sv[-1], "seconds_per_step": sum(secs) / len(secs)},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "pairings": cpu_pairing_run(max(1024, 32 * threads), threads),
            "gpu_launches": 0}
    print(json.dumps(line))
    return 0


def dump_outputs(path: str, arrays: dict) -> None:
    """--dump-outputs: each array of wire bytes as path/<name>.npy, one float32 per byte (0..255, exact), so that two builds
    run with the same arguments (hence the same seeded inputs) can be compared output for output."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, raw in arrays.items():
        np.save(os.path.join(path, name + ".npy"), np.frombuffer(raw, dtype=np.uint8).astype(np.float32))


# ------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from kyber_b200 import Comm, Engine, workload as wl
    from oracle import bls12381 as o

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"          # keep stdout to the one JSON line (NCCL prints its version banner there)
        dist.init_process_group("nccl", device_id=dev)

    # BASELINE.json configs[4] (C5) is 2^24 pairs over 8 GPUs = 2^21 per GPU; configs[1] (C2) is 2^20 on one GPU (also used at 2 and 4)
    log_n = LOG_N if "B2K_BENCH_LOGN" in os.environ else (21 if world == 8 else 20)
    n = 1 << log_n
    eng = Engine(local)
    stream = torch.cuda.current_stream()
    eng.set_stream(stream.cuda_stream)

    # ---- synthetic inputs (seed b2k/c2; rank r owns counters [r*n, (r+1)*n)) --------------------
    a = wl.prng_scalars("b2k/c2-a", n, wl.R_BLS12381, rank * n)
    s = wl.prng_scalars("b2k/c2", n, wl.R_BLS12381, rank * n)
    sb = wl.scalars_to_bytes(s)
    h_scal = torch.frombuffer(bytearray(sb), dtype=torch.uint8).pin_memory()
    h_a = torch.frombuffer(bytearray(wl.scalars_to_bytes(a)), dtype=torch.uint8)
    d_a = h_a.to(dev)
    d_gen = torch.frombuffer(bytearray(wl.G1_BLS12381_AFFINE), dtype=torch.uint8).to(dev).repeat(n)
    d_pts = torch.empty(n * 96, dtype=torch.uint8, device=dev)
    eng.call_dev("b2k_bls12381_g1_mul_batch_affine_dev", n, d_a.data_ptr(), d_gen.data_ptr(), d_pts.data_ptr())
    torch.cuda.synchronize()
    del d_gen, d_a
    h_pts = d_pts.cpu().pin_memory()
    # sample-check the generated points against the oracle
    for i in (0, n // 3, n - 1):
        assert bytes(h_pts[96 * i:96 * i + 96].tolist()) == o.g1_to_affine_bytes(o.g1_mul(a[i])), "bad input point"
    d_scal = h_scal.to(dev)
    d_final = torch.zeros(64, dtype=torch.uint8, device=dev)
    my_dot = wl.dot_mod(s, a, o.R)

    # NC independent steps may be in flight: each has its own context (CUDA stream + scratch arena), so the
    # serial tail of one MSM (bucket reduction, Horner) runs under the bucket-accumulate of the next one.
    NC = max(1, args.contexts)
    streams = [stream] + [torch.cuda.Stream(device=dev) for _ in range(NC - 1)]
    engines = [eng]
    for st in streams[1:]:
        e2 = Engine(local)
        e2.set_stream(st.cuda_stream)
        engines.append(e2)
    finals = [d_final] + [torch.zeros(64, dtype=torch.uint8, device=dev) for _ in range(NC - 1)]

    # ---- multi-GPU: the sharded MSM lives in the library (include/b2kyber.h: b2k_comm_*, b2k_bls12381_g1_msm_sharded_*).
    # One communicator per in-flight context; "peer" = slabs mapped with CUDA IPC, the fused reduction pulls the partial buckets
    # over NVLink; "nccl" = the same exchange through ncclSend/ncclRecv + ncclAllGather issued by the library.
    comms = {"peer": [], "nccl": []}
    xplan = eng.bls12381_g1_msm_bucket_plan(n)
    XC, XW, XNB, XEB = xplan["c"], xplan["W"], xplan["buckets_per_window"], xplan["bucket_bytes"]
    can_exchange = world > 1 and XW % world == 0
    if world > 1:
        for e in engines:
            c = Comm(e, world, rank)
            blobs = [None] * world
            dist.all_gather_object(blobs, c.export())
            c.connect(b"".join(blobs))
            comms["peer"].append(c)
        if can_exchange and not os.environ.get("B2K_SKIP_NCCL"):
            for e in engines:
                c = Comm(e, world, rank)
                ids = [Comm.nccl_unique_id(e.lib) if rank == 0 else None]
                dist.broadcast_object_list(ids, src=0)
                c.use_nccl(ids[0])
                comms["nccl"].append(c)
    # headline shape of the multi-GPU step: the partial-bucket exchange north_star names, on the peer transport
    mode = {"shape": 0 if (can_exchange and args.exchange == "buckets") else 1, "transport": "peer"}

    def step_device(k: int = 0):
        """one pass of the hot path, inputs resident in HBM, issued on context k % NC"""
        j = k % NC
        if world == 1:
            engines[j].call_dev("b2k_bls12381_g1_msm_dev", n, d_scal.data_ptr(), d_pts.data_ptr(), finals[j].data_ptr())
        else:
            comms[mode["transport"]][j].msm_sharded_dev(n, d_scal.data_ptr(), d_pts.data_ptr(), finals[j].data_ptr(), mode["shape"])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(steps: int, warm: int):
        """device time of `steps` steps issued round-robin on the NC contexts (max over the contexts' end events)"""
        for k in range(warm * NC):
            step_device(k)
        barrier()
        ev0 = torch.cuda.Event(enable_timing=True)
        ends = [torch.cuda.Event(enable_timing=True) for _ in range(NC)]
        barrier()
        ev0.record(stream)                   # every stream is idle here (barrier above)
        for k in range(steps):
            step_device(k)
        for st, ev in zip(streams, ends):
            ev.record(st)
        barrier()
        return max(ev0.elapsed_time(ev) for ev in ends)

    # ---- device-resident timing --------------------------------------------------------------------
    for k in range(max(args.warmup, 3) * NC):
        step_device(k)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    launches0 = sum(e.launch_count() for e in engines)
    acc_ms = []
    dev_ms = timed(args.steps, 0)
    launches = sum(e.launch_count() for e in engines) - launches0
    head_got = bytes(finals[(args.steps - 1) % NC][:48].cpu().tolist())
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, {"msm_result": head_got})
    # the other exchange shapes / transports, timed the same way (all reported; --exchange picks the headline one)
    alts = {}
    if world > 1:
        variants = [("result_exchange_peer", 1, "peer")]
        if can_exchange:
            variants.append(("bucket_exchange_peer", 0, "peer"))
            if comms["nccl"]:
                variants.append(("bucket_exchange_nccl", 0, "nccl"))
        head = dict(mode)
        for name, shape, transport in variants:
            if shape == head["shape"] and transport == head["transport"]:
                alts[name] = (dev_ms / args.steps, head_got)
                continue
            mode.update(shape=shape, transport=transport)
            ms = timed(args.steps, 3) / args.steps
            alts[name] = (ms, bytes(finals[(args.steps - 1) % NC][:48].cpu().tolist()))
        mode.update(head)
    # the same K steps on ONE context (no overlap): single-MSM latency
    ev_a, ev_b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev_a.record(stream)
    for _ in range(min(args.steps, 5)):
        step_device(0)
    ev_b.record(stream)
    barrier()
    serial_ms = ev_a.elapsed_time(ev_b) / min(args.steps, 5)
    # stage timings of the last local MSM (CUDA events recorded on the same stream inside the library)
    for _ in range(3):
        eng.call_dev("b2k_bls12381_g1_msm_dev", n, d_scal.data_ptr(), d_pts.data_ptr(), d_final.data_ptr())
        acc_ms.append(eng.last_timings())
    barrier()
    sustained = None
    # ---- end-to-end through the host C ABI (pinned host buffers) -----------------------------------
    hs_ptr, hp_ptr = h_scal.data_ptr(), h_pts.data_ptr()
    h_results = [torch.zeros(64, dtype=torch.uint8).pin_memory() for _ in range(NC)]
    h_res = h_results[0]
    e2e_comms = comms["peer"] if (world > 1 and can_exchange) else None

    def e2e_submit(k: int, NE: int):
        j = k % NE
        e = engines[j]
        if world == 1:
            e._check(e.lib.b2k_bls12381_g1_msm_async(e.h, n, ctypes.c_void_p(hs_ptr), ctypes.c_void_p(hp_ptr),
                                                     ctypes.c_void_p(h_results[j].data_ptr())))
        else:                                    # the SHARDED MSM from host buffers: H2D of the shard, buckets, exchange, sum, D2H
            e2e_comms[j].msm_sharded_async(n, hs_ptr, hp_ptr, h_results[j].data_ptr())

    e2e_status = []

    def e2e_collect(k: int, NE: int):
        e = engines[k % NE]
        e._check(e.lib.b2k_wait(e.h))
        e2e_status.append(bytes(h_results[k % NE][:48].tolist()))

    have_e2e = world == 1 or e2e_comms is not None
    e2e_ms = e2e_blocking_ms = 0.0
    NE = max(1, min(int(os.environ.get("B2K_E2E_INFLIGHT", str(NC))), NC))
    if have_e2e:
        for _ in range(2):
            e2e_submit(0, 1); e2e_collect(0, 1)
        barrier()
        # (a) one caller, blocking back to back: what a strictly synchronous user of the C ABI sees
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(min(args.steps, 5)):
            e2e_submit(0, 1); e2e_collect(0, 1)
        e1.record(stream)
        barrier()
        e2e_blocking_ms = e0.elapsed_time(e1) / min(args.steps, 5)
        # (b) the asynchronous entry point on NE contexts used in turn by ONE host thread: submit step k on context k % NE (H2D of
        #     scalars+points, MSM [+ exchange], D2H of the result, all enqueued), collect step k-NE first.  Every step still moves
        #     its inputs host->device and its result device->host inside the timed region.  Timed on the device.
        for _ in range(2):
            for k in range(NE):
                e2e_submit(k, NE)
            for k in range(NE):
                e2e_collect(k, NE)
        barrier()
        del e2e_status[:]
        ev_start = torch.cuda.Event(enable_timing=True)
        ev_ends = [torch.cuda.Event(enable_timing=True) for _ in range(NE)]
        ev_start.record(streams[0])
        for k in range(args.steps):
            if k >= NE:
                e2e_collect(k - NE, NE)
            e2e_submit(k, NE)
        for j in range(NE):
            ev_ends[j].record(streams[j])
        for k in range(max(0, args.steps - NE), args.steps):
            e2e_collect(k, NE)
        barrier()
        e2e_ms = max(ev_start.elapsed_time(ev) for ev in ev_ends)
    clocks = sampler.finish() if rank == 0 else None

    # ---- correctness of what was timed ---------------------------------------------------------------
    if world > 1:
        dots = [None] * world
        dist.all_gather_object(dots, my_dot)
        total_dot = sum(dots) % o.R
    else:
        total_dot = my_dot
    want = o.g1_compress(o.g1_mul(total_dot))
    assert head_got == want, "device MSM result differs from the oracle"
    if have_e2e:
        assert bytes(h_res[:48].tolist()) == want, "e2e MSM result differs from the oracle"
        assert e2e_status and all(x == want for x in e2e_status), "an asynchronous e2e step returned a wrong result"
    for name, (_, got_alt) in alts.items():
        assert got_alt == want, f"multi-GPU variant {name} disagrees with the oracle"

    # ---- max over ranks ---------------------------------------------------------------------------------
    names = sorted(alts)
    t = torch.tensor([dev_ms, e2e_ms, e2e_blocking_ms, serial_ms] + [alts[k][0] for k in names], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms, e2e_blocking_ms, serial_ms = (float(t[i]) for i in range(4))
    alt_ms = {k: float(t[4 + i]) for i, k in enumerate(names)}

    if rank == 0:
        ms_step = dev_ms / args.steps
        value = world * n / (ms_step * 1e-3)
        tm = [sum(x[i] for x in acc_ms) / len(acc_ms) for i in range(len(acc_ms[0]))]
        plan = eng.last_msm_plan()                                         # what the timed MSMs actually ran with
        c_bits = plan["c"]
        peak, peak_src = load_peaks()
        cfg_name = ("BASELINE.json configs[4] (C5): 2^24 pairs sharded over 8 GPUs" if (world == 8 and log_n == 21) else
                    "BASELINE.json configs[1] (C2)" + (" per GPU" if world > 1 else ""))
        if world == 1:
            xdesc = "none"
        elif mode["shape"] == 0:
            xdesc = (f"partial buckets ({XW * XNB * XEB} B per rank) left in the rank's exchange slab; rank g's fused add+reduce kernel PULLS "
                     f"windows [g W/G, (g+1) W/G) of every rank over NVLink (CUDA-IPC-mapped peer memory, device-side flag words), pushes "
                     f"{XW // world} window sums to every peer, Horner on every rank; no host-issued collective")
        else:
            xdesc = "every rank finishes its MSM, pushes its 96-byte result into every peer's slab, adds the N results"
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
                "config": {"workload": f"BLS12-381 G1 MSM, 2^{log_n} random (scalar,point) pairs per GPU ({cfg_name}); seed b2k/c2",
                           "pairs_per_gpu": n, "pairs_total": n * world,
                           "parallelism": f"shard{world}" if world > 1 else "single",
                           "l2": "no flush: each step streams >400 MB (128 MiB inputs + sort + buckets) > 126 MB L2",
                           "exchange": xdesc,
                           "steps_in_flight": NC,
                           "overlap": f"{NC} independent steps in flight on {NC} contexts/streams; "
                                      "single_step_latency_ms is one step alone"},
                "single_step_latency_ms": serial_ms,
                "gpu_launches": int(launches),
                "clocks": clocks,
                "stages_ms": dict(zip(["load", "digits_hist", "scan", "scatter", "accumulate", "reduce_chunks",
                                       "window_sum", "final", "pipeline", "fixup", "accumulate_affine_rounds"],
                                      [round(x, 4) for x in tm])),
                "msm_plan": plan}
        if have_e2e:
            e2e_value = world * n / (e2e_ms / args.steps * 1e-3)
            line["e2e"] = {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": n * 128, "d2h_bytes_per_step": 52,
                           "ms_per_step": e2e_ms / args.steps, "callers": 1, "steps_in_flight": NE,
                           "blocking_ms_per_step": e2e_blocking_ms,
                           "note": ("b2k_bls12381_g1_msm_async + b2k_wait" if world == 1 else
                                    "b2k_bls12381_g1_msm_sharded_async + b2k_wait (the SHARDED MSM: H2D of the rank's shard, partial buckets, "
                                    "the exchange over peer memory, the sum of all ranks, D2H on every rank)") +
                                   f" on {NE} contexts used in turn by one host thread per rank (pinned host buffers; H2D of all inputs and "
                                   "D2H of the result inside the timed region every step; h2d/d2h bytes are per rank); "
                                   "blocking_ms_per_step = submit + wait back to back on one context"}
        if world > 1:
            line["multi_gpu_exchange"] = {
                "ms_per_step": alt_ms, "headline": ("bucket_exchange_peer" if mode["shape"] == 0 else "result_exchange_peer"),
                "bucket_exchange_bytes_pulled_per_rank": XW * XNB * XEB * (world - 1) // world if can_exchange else None,
                "note": "same sharded MSM, same bytes out, all inside the library (b2k_bls12381_g1_msm_sharded_dev): *_peer = exchange slabs mapped "
                        "with CUDA IPC, device-side flags, the fused add+reduce kernel reads the peers' buckets over NVLink; bucket_exchange_nccl = "
                        "the same exchange as grouped ncclSend/ncclRecv (all-to-all) + ncclAllGather issued by the library (libnccl.so.2 via dlopen); "
                        "result_exchange = every rank finishes its own MSM and the 96-byte results travel"}
        if c_bits:
            nv = n * (2 if plan["glv"] else 1)                            # pairs after the endomorphism split
            adds = nv * plan["W"]                                         # bucket additions (SURVEY.md 8(d): 16 per input pair at c = 16)
            nbuckets = plan["W"] * plan["buckets_per_window"]
            alg_bytes = adds * 100 + nbuckets * 144                       # SURVEY.md 8(d): 100 B per addition + 144 B per bucket
            acc = tm[4] * 1e-3
            R = plan["affine_rounds"]
            left = adds / (1 << R) + (nbuckets if R else 0)               # operands the XYZZ slices still see after R halvings
            products = (adds - left) * 6 + left * 10                      # affine addition 6, mixed XYZZ addition 10 field products
            traffic = None
            tp = os.path.join(ROOT, "profiles", "accumulate_traffic.json")
            if os.path.exists(tp) and log_n == 20:
                try:
                    traffic = json.load(open(tp)).get("dram_bytes_per_launch")
                except Exception:
                    traffic = None
            kern = (f"bucket-accumulate pass: k_pt_forward/k_pt_invert/k_pt_backward x{R} (batched affine additions) + k_msm_accumulate_slices_direct"
                    if R else "k_msm_accumulate_slices")
            line["roofline"] = {"bound": "hbm", "kernel": kern, "achieved": alg_bytes / acc / 1e9,
                                "peak": peak, "unit": "GB/s", "frac": alg_bytes / acc / 1e9 / peak,
                                "traffic": traffic, "peak_source": peak_src,
                                "algorithmic_bytes": alg_bytes, "kernel_ms": tm[4], "window_bits": c_bits,
                                "affine_rounds_ms": tm[10] if len(tm) > 10 else None,
                                "note": "integer-ALU bound pass (SURVEY.md F9): see `integer_roofline` and DESIGN.md section 4; "
                                        "`traffic` is the ncu DRAM bytes of the whole pass (all its launches) for one 2^20 MSM "
                                        "(profiles/accumulate_traffic.json, captured with the same kernels)",
                                "integer_roofline": {
                                    "bound": "fma-heavy pipe (IMAD.WIDE, 4 cycles per warp instruction)",
                                    "achieved": products / acc, "peak": 3.04e10, "unit": "381-bit Montgomery products/s",
                                    "frac": products / acc / 3.04e10,
                                    "peak_source": "measured: tools/probe/fpmul_probe.cu on B200 (profiles/r01_pipe_probes.txt)",
                                    "work": f"{int(adds - left)} affine additions x 6 + {int(left)} mixed XYZZ additions x 10 field products "
                                            "(operand counts after the rounds estimated as adds / 2^R + buckets); the pass did the work of "
                                            f"{adds} XYZZ additions (x 10) of the previous design",
                                    "xyzz_equivalent_frac": adds * 10 / acc / 3.04e10}}
        if world == 1 and not os.environ.get("B2K_SKIP_PAIRINGS"):
            line["independent_muls"] = gpu_mul_batch_run(eng, torch, dev, d_scal, d_pts, n, max(2, min(args.steps, 3)), s, a)
            line["pairings"] = gpu_pairing_run(eng, torch, dev, 1 << 16, max(2, min(args.steps, 5)))
            line["bls_verify"] = gpu_verify_run(eng, torch, dev, 1 << 16, max(2, min(args.steps, 3)))
        if world == 1 and not os.environ.get("B2K_SKIP_CPU_BASELINE"):
            threads = best_cpu_threads()
            line["cpu_baseline"] = cpu_reference_run(1 << 16, threads)
            line["cpu_baseline"]["logical_cpus"] = os.cpu_count()
            if "pairings" in line:
                line["pairings"]["cpu_baseline"] = cpu_pairing_run(max(1024, 32 * threads), threads)
        if world == 1 and not os.environ.get("B2K_SKIP_SECTIONS"):
            threads = best_cpu_threads()
            line["recover_commit"] = section_recover_commit(eng, torch, 5, threads)
            line["bdn_aggregate"] = section_bdn_aggregate(eng, torch, 3, threads)
            line["ed25519"] = section_ed25519(eng, torch, 10)
        # a sustained run (seconds, not a burst): the headline step for >= 3 s with its own clock sample, LAST so that the power
        # state it leaves behind does not leak into the other sections
        if world == 1 and not os.environ.get("B2K_SKIP_SUSTAINED"):
            est = dev_ms / args.steps
            ks = max(args.steps, int(3000.0 / est) + 1)
            samp2 = ClockSampler(local)
            samp2.start()
            time.sleep(0.2)
            sus_ms = timed(ks, 0)
            line["sustained"] = {"value": n * ks / (sus_ms * 1e-3), "unit": UNIT, "steps": ks, "seconds": sus_ms * 1e-3,
                                 "ms_per_step": sus_ms / ks, "clocks": samp2.finish()}
        print(json.dumps(line))
    if world > 1:
        barrier()
        for cs in comms.values():
            for c in cs:
                c.close()
        dist.destroy_process_group()
    return 0


def main():
    # stdout carries exactly ONE JSON line: libraries (NCCL's version banner, torch.distributed) write to fd 1 too, so everything
    # else goes to stderr and the line is written to the saved descriptor at the end
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(os.dup(2), "w")
    buf = []
    import builtins
    orig_print = builtins.print

    def capture(*a, **k):
        if k.get("file") in (None, sys.stdout) and len(a) == 1 and isinstance(a[0], str) and a[0].startswith("{"):
            buf.append(a[0])
        else:
            orig_print(*a, **k)
    builtins.print = capture
    try:
        rc = _main()
    finally:
        builtins.print = orig_print
        for line in buf[-1:]:
            os.write(real_stdout, (line + "\n").encode())
    return rc


def _main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--exchange", default="buckets", choices=["result", "buckets"],
                    help="multi-GPU exchange shape of the headline step (the other one is timed and reported beside it)")
    ap.add_argument("--contexts", type=int, default=4, help="independent steps in flight (streams); 1 = strictly serial")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the MSM result of the last timed step (48-byte compressed G1 point) "
                         "to DIR/msm_result.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "reference":
        return run_reference_arm(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())

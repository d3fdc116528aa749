"""GPU parity of the Pippenger MSM and the Point.Mul batch on every group they are built for besides BLS12-381 G1 --
BLS12-381 G2, bn254 G1 and G2, bn256 G1 and G2 -- plus the BLS12-381 entry points no other test reaches: the MSM with the
sum in operand form (what the Go adapter's groupBls.MSM calls), the device-pointer MSM / Point.Mul calls with their status
reported at b2k_wait, and the chunked host-to-device upload of a large G1 MSM.

The pipeline (msm_host.cuh, msm.cuh, kernels.cuh) and scalar_mul_w4 are templates over the curve: a slip in one instance
shows only on that group, at the window width, slice length, reduction scheme or scalar distribution where it lives.  The
expected value is always the Python oracle (oracle/bls12381.py, bn254.py, bn254_pairing.py, bn256.py): the sum of
per-element products for small inputs, and for large ones the known discrete logs
    sum s_i (a_i G) = ((sum s_i a_i) mod r) G,
with the points a_i G made by the engine's fixed-base Point.Mul and a sample of them re-checked against the oracle.
Results are compared as wire bytes.
"""
import contextlib
import functools
import random
from dataclasses import dataclass
from typing import Callable, Optional

import pytest

from kyber_b200 import B2KError
from kyber_b200 import workload as wl
from oracle import bls12381 as ob
from oracle import bn254 as o254
from oracle import bn254_pairing as o254p
from oracle import bn256 as o256

pytestmark = pytest.mark.gpu


# ---- one row per group -------------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class Group:
    name: str
    order: int
    p: int                               # base field modulus
    mul: str                             # Point.Mul batch, results in wire form
    mul_op: str                          # Point.Mul batch, results in operand form (points fed back into the MSM)
    msm: str
    op_bytes: int                        # operand point
    res_bytes: int                       # wire result
    coord_bytes: int                     # one base-field coordinate inside an operand
    o_mul: Callable                      # oracle (k, pt) -> k pt
    o_add: Callable
    gen: object
    enc_op: Callable                     # oracle point -> operand bytes
    enc_res: Callable                    # oracle point -> wire result bytes
    o_neg: Optional[Callable]            # None: -P = (order - 1) P
    range_checked: bool                  # operand coordinates >= p are refused (include/b2kyber.h: BLS12-381, bn254)


GROUPS = [
    Group("bls12381_g2", ob.R, ob.P, "b2k_bls12381_g2_mul_batch", "b2k_bls12381_g2_mul_batch_affine", "b2k_bls12381_g2_msm",
          192, 96, 48, ob.g2_mul, ob.g2_add, ob.G2, ob.g2_to_affine_bytes, ob.g2_compress, ob.g2_neg, True),
    Group("bn254_g1", o254.ORDER, o254.P, "b2k_bn254_g1_mul_batch", "b2k_bn254_g1_mul_batch", "b2k_bn254_g1_msm",
          64, 64, 32, o254.g1_mul, o254.g1_add, o254.G1, o254.g1_marshal, o254.g1_marshal, o254.g1_neg, True),
    Group("bn254_g2", o254p.ORDER, o254p.P, "b2k_bn254_g2_mul_batch", "b2k_bn254_g2_mul_batch", "b2k_bn254_g2_msm",
          128, 128, 32, o254p.g2_mul, o254p.g2_add, o254p.G2, o254p.g2_marshal, o254p.g2_marshal, o254p.g2_neg, True),
    Group("bn256_g1", o256.ORDER, o256.P, "b2k_bn256_g1_mul_batch", "b2k_bn256_g1_mul_batch", "b2k_bn256_g1_msm",
          64, 64, 32, o256.g1_mul, o256.g1_add, o256.G1, o256.g1_marshal, o256.g1_marshal, None, False),
    Group("bn256_g2", o256.ORDER, o256.P, "b2k_bn256_g2_mul_batch", "b2k_bn256_g2_mul_batch", "b2k_bn256_g2_msm",
          128, 128, 32, o256.g2_mul, o256.g2_add, o256.G2, o256.g2_marshal, o256.g2_marshal, None, False),
]
BLS_G1 = Group("bls12381_g1", ob.R, ob.P, "b2k_bls12381_g1_mul_batch", "b2k_bls12381_g1_mul_batch_affine", "b2k_bls12381_g1_msm",
               96, 48, 48, ob.g1_mul, ob.g1_add, ob.G1, ob.g1_to_affine_bytes, ob.g1_compress, ob.g1_neg, True)
by_group = pytest.mark.parametrize("g", GROUPS, ids=[g.name for g in GROUPS])

N_CACHED = (1 << 17) + 5                 # the largest MSM of the automatic-plan test; every smaller MSM uses a prefix


def _mul(g, k, pt):
    return g.o_mul(k % g.order, pt)


def _neg(g, pt):
    return g.o_neg(pt) if g.o_neg else _mul(g, g.order - 1, pt)


def _sum(g, pts):
    return functools.reduce(g.o_add, pts, None)


def _sb(ks) -> bytes:
    return b"".join(k.to_bytes(32, "big") for k in ks)


def _msm(engine, g, ks, pts: bytes) -> bytes:
    return engine.call_host(g.msm, len(ks), _sb(ks), pts, g.res_bytes)


def _mul_batch(engine, g, ks, pts: bytes, operand_form=False) -> bytes:
    name, width = (g.mul_op, g.op_bytes) if operand_form else (g.mul, g.res_bytes)
    return engine.call_host(name, len(ks), _sb(ks), pts, width * len(ks))


def _known_log_want(g, s, a) -> bytes:
    return g.enc_res(_mul(g, wl.dot_mod(s, a, g.order), g.gen))


@contextlib.contextmanager
def _knobs(engine, c=0, L=0, one_thread_per_bucket=False, groups=1, reduce=(0, 0, 0)):
    """MSM context knobs for the body of a with-block; every one is back at its default afterwards, also on failure"""
    try:
        engine.set_msm_window(c)
        engine.set_msm_slice(L)
        engine.set_msm_variant(one_thread_per_bucket)
        engine.set_msm_groups(groups)
        engine.set_msm_reduce(*reduce)
        yield
    finally:
        engine.set_msm_window(0)
        engine.set_msm_slice(0)
        engine.set_msm_variant(False)
        engine.set_msm_groups(1)
        engine.set_msm_reduce(0, 0, 0)


_POINTS = {}


def _points(engine, g):
    """(a, operand bytes of a_i G) for N_CACHED pairs, made once per group by the engine's fixed-base Point.Mul.  The a_i put
    equal operands (10, 11, 12), a P / -P pair (20, 21) and an operand at infinity (30) into the set; those and a sample of
    the rest are re-checked against the oracle."""
    if g.name not in _POINTS:
        a = wl.prng_scalars("b2k/curves-a-" + g.name, N_CACHED, g.order)
        a[10] = a[11] = a[12]
        a[20] = g.order - a[21]
        a[30] = 0
        pts = engine.call_host(g.mul_op, N_CACHED, _sb(a), g.enc_op(g.gen) * N_CACHED, g.op_bytes * N_CACHED)
        w = g.op_bytes
        for i in (0, 10, 12, 20, 21, 30, 127, 128, 2999, N_CACHED // 2, N_CACHED - 1):
            assert pts[w * i:w * i + w] == g.enc_op(_mul(g, a[i], g.gen)), (g.name, i)
        _POINTS[g.name] = (a, pts)
    return _POINTS[g.name]


# ---- 1. exceptional buckets at every window width -------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _exceptional_case(name):
    """n = 37 pairs: P + P and P + (-P) under one scalar (same bucket in every window), an operand at infinity, scalars 0,
    order - 1, order - 2; the expected sum is the oracle's sum of the 37 products"""
    g = next(x for x in GROUPS if x.name == name)
    rng = random.Random("b2k/curves-exc-" + name)
    n = 37
    ks = [rng.randrange(g.order) for _ in range(n)]
    pts = [_mul(g, rng.randrange(1, 1 << 64), g.gen) for _ in range(n)]
    pts[1], ks[1] = pts[0], ks[0]
    pts[3], ks[3] = _neg(g, pts[2]), ks[2]
    pts[4] = None
    ks[5] = 0
    ks[6] = g.order - 1
    ks[7] = g.order - 2
    want = g.enc_res(_sum(g, [_mul(g, k, pt) for k, pt in zip(ks, pts)]))
    return ks, b"".join(g.enc_op(pt) for pt in pts), want


@by_group
@pytest.mark.parametrize("c", [0] + list(range(4, 17)), ids=lambda c: "c%d" % c)
def test_exceptional_buckets_every_window(engine, g, c):
    ks, pts, want = _exceptional_case(g.name)
    with _knobs(engine, c=c):
        got = _msm(engine, g, ks, pts)
        if c:
            assert engine.last_msm_plan()["c"] == c
    assert got == want


# ---- 2. skewed scalar distributions ---------------------------------------------------------------------------------------
def _skewed_scalars(g, dist, n):
    rng = random.Random("b2k/curves-skew-%s-%s" % (g.name, dist))
    if dist == "equal":                  # one bucket per window holds all n entries: the fix-up of big buckets
        s = [g.order * 5 // 7] * n
    elif dist == "small":                # empty upper windows
        s = [rng.randrange(1 << 20) for _ in range(n)]
    elif dist == "two_values":
        s = [rng.choice([1, g.order - 1]) for _ in range(n)]
    elif dist == "bdn128":               # sign/bdn coefficients c_i + 1
        s = [rng.randrange(1 << 128) + 1 for _ in range(n)]
    else:                                # "high" (bn256): every scalar in [2^255, order), top digit of the 256-bit plan set
        s = [(1 << 255) + rng.randrange(g.order - (1 << 255)) for _ in range(n)]
    s[10] = s[11] = s[12]                # equal operands 10..12 and the pair P, -P (20, 21) meet inside the same buckets
    s[20] = s[21]
    return s


SKEW_CASES = [(g, d) for g in GROUPS for d in ("equal", "small", "two_values", "bdn128") + (("high",) if g.name.startswith("bn256") else ())]


@pytest.mark.parametrize("g,dist", SKEW_CASES, ids=["%s-%s" % (g.name, d) for g, d in SKEW_CASES])
def test_skewed_scalar_distributions(engine, g, dist):
    n = 3000
    a, pts = _points(engine, g)
    a, pts = a[:n], pts[:g.op_bytes * n]
    s = _skewed_scalars(g, dist, n)
    want = _known_log_want(g, s, a)
    for c, L in ((0, 0), (16, 0), (8, 3), (11, 1), (4, 1)):
        with _knobs(engine, c=c, L=L):
            got = _msm(engine, g, s, pts)
            plan = engine.last_msm_plan()
        assert got == want, (dist, c, L)
        if dist == "equal":              # the full bucket spans more than 64 slices: k_msm_fixup_big has work
            assert n > 64 * plan["slice_len"], plan
    with _knobs(engine, one_thread_per_bucket=True):
        assert _msm(engine, g, s, pts) == want, "one thread per bucket"
    with _knobs(engine, c=8, groups=4):  # overlapped tail: windows in 4 groups, reduction on the second stream
        got = _msm(engine, g, s, pts)
        assert engine.last_msm_plan()["W"] >= 8
    assert got == want, "overlapped tail"


# ---- 3. automatic plans across sizes ----------------------------------------------------------------------------------------
@by_group
def test_automatic_plans_across_sizes(engine, g):
    a, pts = _points(engine, g)
    for n in (1, 3, 129, 1000, 20001, N_CACHED):
        s = wl.prng_scalars("b2k/curves-auto-%s-%d" % (g.name, n), n, g.order)
        got = _msm(engine, g, s, pts[:g.op_bytes * n])
        assert got == _known_log_want(g, s, a[:n]), n
    plan = engine.last_msm_plan()         # the largest size: wide windows and the two-level bucket reduction
    assert plan["c"] >= 13 and plan["reduce_levels"] == 2, plan


def test_automatic_plan_split_window_sum_bn254_g1(engine):
    """n = 2^18 + 3 on bn254 G1: automatic c >= 14, two-level reduction with so many partials per window that the window
    sum runs in sub-blocks (msm_host.cuh: window_sum_split)"""
    g = GROUPS[1]
    n = (1 << 18) + 3
    a = wl.prng_scalars("b2k/curves-big-a", n, g.order)
    s = wl.prng_scalars("b2k/curves-big-s", n, g.order)
    pts = _mul_batch(engine, g, a, g.enc_op(g.gen) * n, operand_form=True)
    for i in (0, n // 3, n - 1):
        assert pts[64 * i:64 * i + 64] == g.enc_op(_mul(g, a[i], g.gen)), i
    assert _msm(engine, g, s, pts) == _known_log_want(g, s, a)
    plan = engine.last_msm_plan()
    m1, m2 = plan["reduce_chunks"] if plan["reduce_levels"] == 2 else (0, 0)
    assert plan["c"] >= 14 and plan["reduce_levels"] == 2, plan
    nb = plan["buckets_per_window"]
    assert nb // m1 + nb // (m1 * m2) >= 1024, plan   # partials per window: window_sum_split cuts them into sub-blocks


# ---- 4. both reduction schemes ------------------------------------------------------------------------------------------------
@by_group
@pytest.mark.parametrize("c", [8, 13, 16], ids=lambda c: "c%d" % c)
def test_reduction_schemes(engine, g, c):
    n = 600
    a, pts = _points(engine, g)
    a, pts = a[:n], pts[:g.op_bytes * n]
    rng = random.Random("b2k/curves-red-%s-%d" % (g.name, c))
    nb = 1 << (c - 1)
    for s in (wl.prng_scalars("b2k/curves-red-" + g.name, n, g.order), [rng.randrange(1 << 128) for _ in range(n)], [g.order - 1] * n):
        want = _known_log_want(g, s, a)
        for levels, m1, m2 in ((0, 0, 0), (1, 0, 0), (2, 0, 0), (2, 2, 8), (2, 8, 2), (2, 16, 16), (2, 1, 4), (2, 4, 1)):
            with _knobs(engine, c=c, reduce=(levels, m1, m2)):
                got = _msm(engine, g, s, pts)
                plan = engine.last_msm_plan()
            assert got == want, (levels, m1, m2)
            assert plan["c"] == c
            if levels:                   # forced two levels fall back to one when m1 m2 does not divide the bucket count
                assert plan["reduce_levels"] == (2 if levels == 2 and nb % ((m1 or 8) * (m2 or 4)) == 0 else 1), (levels, m1, m2, plan)


# ---- 5. Point.Mul batch at the edges of the signed radix-16 recoding ---------------------------------------------------------
def _mul_edge_scalars(g):
    r = g.order
    ks = [0, 1, 2, 7, 8, 9, 15, 16, 17, 0x88, 0x78, 0xff, 0x100, (1 << 32) - 1, 1 << 32, (1 << 64) - 8, 1 << 128, r - 1, r - 2,
          r - 7, r - 8, r - 9, r - 16, (r - 1) // 2, (r + 1) // 2]
    for d in "87f":                      # runs of 8s / 7s / fs: every digit at the edge of its range, carries through many digits
        for length in (8, 16, 31, 32, 33, 48, 62, 63, 64):
            v = int(d * length, 16)
            if v < r:
                ks.append(v)
    if r.bit_length() == 256:            # bn256: the top digit carries into the 65th digit
        rng = random.Random("b2k/curves-mul-high")
        ks += [1 << 255, (1 << 255) + 1, (1 << 255) + int("8" * 63, 16), r - 3, r - 0x80]
        ks += [(1 << 255) + rng.randrange(r - (1 << 255)) for _ in range(12)]
    return ks


@by_group
def test_mul_batch_recoding_edges(engine, g):
    n = 129                              # the second 128-thread block holds one element
    rng = random.Random("b2k/curves-mul-" + g.name)
    edges = _mul_edge_scalars(g)
    ks = edges + [rng.randrange(1 << 32) for _ in range(n - len(edges) - 1)] + [g.order - 1]
    assert len(ks) == n
    bases = [_mul(g, rng.randrange(1, 1 << 64), g.gen) for _ in range(7)] + [None]     # the 8th operand is at infinity
    pts = [bases[i % 8] for i in range(n)]
    pts[n - 1] = bases[0]
    pb = b"".join(g.enc_op(pt) for pt in pts)
    out = _mul_batch(engine, g, ks, pb)
    out_op = _mul_batch(engine, g, ks, pb, operand_form=True) if g.mul_op != g.mul else None
    for i in range(n):
        want = _mul(g, ks[i], pts[i])
        assert out[g.res_bytes * i:g.res_bytes * (i + 1)] == g.enc_res(want), (i, hex(ks[i]))
        if out_op is not None:
            assert out_op[g.op_bytes * i:g.op_bytes * (i + 1)] == g.enc_op(want), (i, hex(ks[i]))


# ---- 6. range and validation --------------------------------------------------------------------------------------------------
def _with_coord(g, op: bytes, idx: int, value: int) -> bytes:
    w = g.coord_bytes
    return op[:w * idx] + value.to_bytes(w, "big") + op[w * (idx + 1):]


@by_group
def test_scalar_range_and_malformed_operands(engine, g):
    pt = _mul(g, 0x1234567, g.gen)
    op = g.enc_op(pt)

    def clean_call():                    # the context carries no stale status after a refused call
        assert _mul_batch(engine, g, [3], op) == g.enc_res(_mul(g, 3, pt))
        assert _msm(engine, g, [3, 5], op * 2) == g.enc_res(_mul(g, 8, pt))

    def refused(code, ks, pts):
        for call in (_mul_batch, _msm):
            with pytest.raises(B2KError) as e:
                call(engine, g, ks, pts)
            assert e.value.code == code, call.__name__
            clean_call()

    refused(-3, [g.order], op)                                        # scalar == order: B2K_ERR_SCALAR_RANGE
    refused(-3, [5, g.order], op * 2)
    assert _mul_batch(engine, g, [g.order - 1], op) == g.enc_res(_neg(g, pt))       # order - 1 is accepted
    assert _msm(engine, g, [g.order - 1, 1], op * 2) == g.enc_res(None)
    last = g.op_bytes // g.coord_bytes - 1                            # the last coordinate: y (its real part on G2)
    y = int.from_bytes(op[-g.coord_bytes:], "big")
    refused(-5, [7], _with_coord(g, op, last, (y + 1) % g.p))         # off the curve: B2K_ERR_POINT
    refused(-5, [7, 9], op + _with_coord(g, op, last, (y + 1) % g.p))
    if g.range_checked:                                               # y + p: the same point mod p, not canonical
        refused(-5, [7], _with_coord(g, op, last, y + g.p))
        refused(-5, [7, 9], op + _with_coord(g, op, 0, int.from_bytes(op[:g.coord_bytes], "big") + g.p))


# ---- 7. BLS12-381 MSM with the sum in operand form ------------------------------------------------------------------------------
AFFINE_MSM = {
    1: (BLS_G1, "b2k_bls12381_g1_msm_affine", ob.g1_decompress),
    2: (GROUPS[0], "b2k_bls12381_g2_msm_affine", ob.g2_decompress),
}


@pytest.mark.parametrize("group", [1, 2], ids=["bls12381_g1", "bls12381_g2"])
def test_msm_affine_output(engine, group):
    g, name, decompress = AFFINE_MSM[group]
    w = g.op_bytes

    def msm_aff(ks, pts):
        return engine.call_host(name, len(ks), _sb(ks), pts, w)

    rng = random.Random("b2k/curves-aff-%d" % group)
    for n in (1, 2):
        ks = [rng.randrange(g.order) for _ in range(n)]
        pts = [_mul(g, rng.randrange(1, g.order), g.gen) for _ in range(n)]
        assert msm_aff(ks, b"".join(g.enc_op(pt) for pt in pts)) == g.enc_op(_sum(g, [_mul(g, k, pt) for k, pt in zip(ks, pts)])), n
    # the Go adapter's Add / Sub / Null cases: unit scalars on (P, P), (P, -P), (P, infinity)
    pt = _mul(g, rng.randrange(1, g.order), g.gen)
    op = g.enc_op(pt)
    assert msm_aff([1, 1], op * 2) == g.enc_op(g.o_add(pt, pt))
    assert msm_aff([1, 1], op + g.enc_op(_neg(g, pt))) == bytes(w)
    assert msm_aff([1, 1], op + bytes(w)) == op
    assert msm_aff([12345, g.order - 12345], op * 2) == bytes(w)
    # n = 1000 with known discrete logs; then the same terms with the last scalar chosen so that the whole sum cancels
    n = 1000
    a = wl.prng_scalars("b2k/curves-aff-a-%d" % group, n, g.order)
    s = wl.prng_scalars("b2k/curves-aff-s-%d" % group, n, g.order)
    pts = engine.call_host(g.mul_op, n, _sb(a), g.enc_op(g.gen) * n, w * n)
    for i in (0, n - 1):
        assert pts[w * i:w * i + w] == g.enc_op(_mul(g, a[i], g.gen)), i
    got = msm_aff(s, pts)
    assert got == g.enc_op(_mul(g, wl.dot_mod(s, a, g.order), g.gen))
    compressed = _msm(engine, g, s, pts)             # the same sum, compressed, decoded
    assert g.enc_op(decompress(compressed, subgroup_check=False)) == got
    s[-1] = -wl.dot_mod(s[:-1], a[:-1], g.order) * pow(a[-1], -1, g.order) % g.order
    assert msm_aff(s, pts) == bytes(w)
    assert _msm(engine, g, s, pts) == g.enc_res(None)


# ---- 8. device-pointer entry points -------------------------------------------------------------------------------------------
G2_ROW, BN254_ROW = GROUPS[0], GROUPS[1]
# name, host-buffer twin, group row, MSM (one result) or Point.Mul (one result per pair), output bytes per result
DEV_CASES = [
    ("b2k_bls12381_g2_msm_dev", "b2k_bls12381_g2_msm", G2_ROW, True, 96),
    ("b2k_bn254_g1_msm_dev", "b2k_bn254_g1_msm", BN254_ROW, True, 64),
    ("b2k_bls12381_g1_msm_affine_dev", "b2k_bls12381_g1_msm_affine", BLS_G1, True, 96),
    ("b2k_bls12381_g1_mul_batch_dev", "b2k_bls12381_g1_mul_batch", BLS_G1, False, 48),
    ("b2k_bls12381_g1_mul_batch_affine_dev", "b2k_bls12381_g1_mul_batch_affine", BLS_G1, False, 96),
    ("b2k_bls12381_g2_mul_batch_affine_dev", "b2k_bls12381_g2_mul_batch_affine", G2_ROW, False, 192),
]


@pytest.mark.parametrize("name,host,g,is_msm,width", DEV_CASES, ids=[c[0] for c in DEV_CASES])
def test_dev_entry_points(engine, name, host, g, is_msm, width):
    import torch
    dev = torch.device("cuda", 0)
    n = 300
    a = wl.prng_scalars("b2k/curves-dev-a-" + g.name, n, g.order)
    s = wl.prng_scalars("b2k/curves-dev-s-" + g.name, n, g.order)
    pts = engine.call_host(g.mul_op, n, _sb(a), g.enc_op(g.gen) * n, g.op_bytes * n)
    out_len = width if is_msm else width * n
    want = engine.call_host(host, n, _sb(s), pts, out_len)
    if is_msm:                                       # the host-buffer twin itself against the oracle
        total = _mul(g, wl.dot_mod(s, a, g.order), g.gen)
        assert want == (g.enc_op(total) if width == g.op_bytes else g.enc_res(total))
    d_s = torch.frombuffer(bytearray(_sb(s)), dtype=torch.uint8).to(dev)
    d_p = torch.frombuffer(bytearray(pts), dtype=torch.uint8).to(dev)
    d_o = torch.zeros(out_len, dtype=torch.uint8, device=dev)
    bad = d_s.clone()
    bad[32 * 7:32 * 8] = torch.frombuffer(bytearray(g.order.to_bytes(32, "big")), dtype=torch.uint8).to(dev)
    torch.cuda.synchronize()                         # torch works on its own stream, the engine on the context's
    engine.wait()                                    # clean slate

    def run(d_scalars):
        d_o.zero_()
        torch.cuda.synchronize()
        engine.call_dev(name, n, d_scalars.data_ptr(), d_p.data_ptr(), d_o.data_ptr())

    run(d_s)
    engine.wait()
    assert d_o.cpu().numpy().tobytes() == want
    run(bad)                                         # accepted at submission ...
    with pytest.raises(B2KError) as e:
        engine.wait()                                # ... reported here
    assert e.value.code == -3
    engine.wait()                                    # cleared
    run(d_s)
    engine.wait()
    assert d_o.cpu().numpy().tobytes() == want


# ---- 9. chunked host-to-device upload of a large BLS12-381 G1 MSM --------------------------------------------------------------
@pytest.mark.parametrize("n", [(1 << 18) + 3, (1 << 18) - 1], ids=["chunked_short_tail", "unchunked"])
def test_g1_msm_chunked_upload(engine, n):
    """n >= 2^18 with the endomorphism split: the inputs are copied in 8 chunks, each prepared as it lands; 2^18 + 3 leaves a
    short last chunk (8 x 32769 > n), 2^18 - 1 stays below the threshold"""
    g = BLS_G1
    a = wl.prng_scalars("b2k/curves-chunk-a", n, g.order)
    s = wl.prng_scalars("b2k/curves-chunk-s", n, g.order)
    pts = engine.bls12381_g1_mul_batch_affine(_sb(a), g.enc_op(g.gen) * n)
    per = (n + 7) // 8
    for i in (0, per - 1, per, 7 * per, n - 1):
        assert pts[96 * i:96 * i + 96] == g.enc_op(_mul(g, a[i], g.gen)), i
    assert engine.bls12381_g1_msm(_sb(s), pts) == _known_log_want(g, s, a)
    assert engine.last_msm_plan()["glv"]

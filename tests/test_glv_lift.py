"""Lifted GLV digits of the throughput MSM (glv.cuh glv_lift_term, the code k_msm_digits runs), on the host.

A lifted geometry splits every fold scalar as k = a - b lambda (mod r) with a, b >= 0 spread over [0, 2^(W c - 1)) by lattice
lifts, and emits the signed c-bit digits of a (on P) and of -b (on phi(P)).  Checked for every window size the geometry model
can pick, with W = ceil(131 / c): the identity mod r, digit bounds, no carry out of the top window, and the top-window load."""
import ctypes
import os
import random
import subprocess

import pytest

import bn254 as bn

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
LAM = 0xB3C4D79D41A917585BFC41088D8DAAA78B17EA66B99C90DD  # phi(P) = [lambda] P
A1 = 0x89D3256894D213E3
B1M = 0x6F4D8248EEB859FC8211BBEB7D4F1128
A2 = 0x6F4D8248EEB859FD0BE4E1541221250B
B2 = A1


@pytest.fixture(scope="module")
def prim(tmp_path_factory):
    """tests/hostlib/glv_harness.cpp, a host build of glv.cuh, compiled into a temporary directory"""
    out = str(tmp_path_factory.mktemp("glv") / "libglv.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I", os.path.join(ROOT, "halo2-verifier_b200", "csrc"),
                    "-x", "c++", os.path.join(HERE, "hostlib", "glv_harness.cpp"), "-o", out], check=True)
    return ctypes.CDLL(out)


def L(v, n=8):
    return (ctypes.c_uint32 * n)(*[(v >> (32 * i)) & 0xFFFFFFFF for i in range(n)])


def lift(prim, k, t, c, W):
    out = (ctypes.c_uint32 * 12)()
    prim.t_glv_lift_term(L(k), t, c, W, out)
    a = sum(out[i] << (32 * i) for i in range(5))
    b = sum(out[5 + i] << (32 * i) for i in range(5))
    return a, b, out[10], out[11]


def signed_digits(v, c, W):
    """msm_emit_digits: signed c-bit digits in (-2^(c-1), 2^(c-1)], the final carry"""
    ds, carry = [], 0
    for w in range(W):
        x = ((v >> (w * c)) & ((1 << c) - 1)) + carry
        if x > 1 << (c - 1):
            ds.append(x - (1 << c))
            carry = 1
        else:
            ds.append(x)
            carry = 0
    return ds, carry


def edge_scalars(rng):
    ks = [0, 1, 2, bn.R - 1, bn.R - 2, LAM, bn.R - LAM, (1 << 127) - 1, (1 << 127) + 1, (1 << 127), (bn.R - 1) // 2]
    # scalars that drive a half to its extremes: k = k1 + k2 lambda for halves at the ends of the proven ranges
    for f1, f2 in ((0, 0), (1, 0), (0, 1), (1, 1)):
        for e1 in (0, 1, 2):
            for e2 in (0, 1, 2):
                k1, k2 = f1 * (A1 + A2) - e1, -f2 * B1M + e2
                ks.append((k1 + k2 * LAM) % bn.R)
                ks.append((f2 * B2 - e1 + (f1 * A2 - e2) * LAM) % bn.R)
    return ks


CS = list(range(4, 16))


def windows(c):
    return (131 + c - 1) // c


def test_lift_ranges_leave_room_at_every_window_size(prim):
    for c in CS:
        _, _, Z, Z2 = lift(prim, 5, 0, c, windows(c))
        cap = 1 << (windows(c) * c - 1)
        assert Z >= 1 and Z2 >= 7, (c, Z, Z2)
        # the proven bounds of glv_lift (glv.cuh) at the ranges chosen
        assert 5 * (A1 + A2) // 4 + 1 + (Z - 1) * A2 + Z2 * A1 <= cap and (4 * Z2 + 5) * B1M // 4 + 1 <= cap, c
    _, _, Z, Z2 = lift(prim, 5, 0, 10, 13)  # 130 bits: little room
    assert Z2 >= 1


@pytest.mark.parametrize("c", CS)
def test_lifted_digits(prim, c):
    """k = sum_w 2^(c w) (d1_w + lambda d2_w) mod r, |d| <= 2^(c-1), no carry out of window W - 1, on 10^4 seeded scalars
    (fewer at the extreme window sizes) and the edge cases, each at several term ids (lifts)"""
    W = windows(c)
    rng = random.Random(100 + c)
    n = 10000 if c in (10, 11, 12, 13) else 1500
    ks = edge_scalars(rng) + [rng.randrange(bn.R) for _ in range(n)]
    for i, k in enumerate(ks):
        for t in ((i, 0xFFFFFFFF - i) if i < 200 else (i * 7919,)):
            a, b, Z, Z2 = lift(prim, k, t & 0xFFFFFFFF, c, W)
            assert (a - b * LAM) % bn.R == k, (hex(k), t)
            da, ca = signed_digits(a, c, W)
            db, cb = signed_digits(b, c, W)
            assert ca == 0 and cb == 0, ("carry out of the top window", hex(k), c)
            assert all(abs(d) <= 1 << (c - 1) for d in da + db)
            tot = sum((x - y * LAM) << (c * w) for w, (x, y) in enumerate(zip(da, db)))
            assert tot % bn.R == k


@pytest.mark.parametrize("c", [10, 11, 12, 13])
def test_top_window_load(prim, c):
    """the lift spreads both halves over the whole window range: the top window's fullest bucket holds at most 2.5x the mean
    of its used-bucket range (seeded sample, ~100 entries per bucket)"""
    W = windows(c)
    B = 1 << (c - 1)
    rng = random.Random(7)
    n = 100 * B // 2
    load = [0] * (B + 1)
    for t in range(n):
        a, b, _, _ = lift(prim, rng.randrange(bn.R), t, c, W)
        for v in (a, b):
            d, _ = signed_digits(v, c, W)
            load[abs(d[-1])] += 1
    mean = 2 * n / B
    assert max(load[1:]) <= 2.5 * mean, (c, max(load[1:]) / mean)

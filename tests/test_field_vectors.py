"""Device field arithmetic of both BN254 fields against exact Python integers (h2v_selftest_field_vectors: raw limbs in and
out).  h2v_selftest_field only compares the PTX path with the portable one, on operands that barely reach the top of each
range; here every operation is checked on the edge classes of its documented domain (field.cuh), their full cross product,
and 10^5 random pairs.  Outputs must be the canonical representative: the kernels compare raw limbs with ==."""
import ctypes
import functools
import random

import pytest

import bn254 as bn

FIELDS = {"Fq": (0, bn.P), "Fr": (1, bn.R)}
OPS = {"mul": 0, "mul_c": 1, "sqr": 2, "sqr_c": 3, "mul_any": 4, "add": 5, "sub": 6, "neg": 7, "from_canonical": 8,
       "to_canonical": 9, "inv": 10, "inv_bin": 11, "from_uniform": 12}
BINARY = {"mul", "mul_c", "mul_any", "add", "sub", "from_uniform"}
RANDOM_PAIRS = 100_000
M32 = 0xFFFFFFFF


def domain(op, p):
    """(bound of a, bound of b): field.cuh specifies mul for a < 2^255, mul_any for any 256-bit a (and b without a limb
    0xFFFFFFFF, see in_domain_b), from_uniform reads a | b as one 512-bit integer; everything else takes reduced operands"""
    if op in ("mul", "mul_c"):
        return 1 << 255, p
    if op == "mul_any":
        return 1 << 256, p
    if op == "from_uniform":
        return 1 << 256, 1 << 256
    return p, p


@functools.lru_cache(maxsize=None)
def r_inv(p):
    return pow(1 << 256, -1, p)


def expected(op, p, a, b):
    R = 1 << 256
    if op in ("mul", "mul_c", "mul_any"):
        return a * b * r_inv(p) % p
    if op in ("sqr", "sqr_c"):
        return a * a * r_inv(p) % p
    if op == "add":
        return (a + b) % p
    if op == "sub":
        return (a - b) % p
    if op == "neg":
        return -a % p
    if op == "from_canonical":
        return a * R % p
    if op == "to_canonical":
        return a * r_inv(p) % p
    if op in ("inv", "inv_bin"):  # Montgomery form in and out: (a/R)^-1 R = R^2 / a; inv(0) = 0
        return 0 if a == 0 else R * R * pow(a, -1, p) % p
    if op == "from_uniform":
        return (a + (b << 256)) * R % p
    raise KeyError(op)


def in_domain_b(op, b):
    """mul_any's right operand must not have a limb 0xFFFFFFFF (field.cuh); its callers pass R^2 and R^3 mod p"""
    return op != "mul_any" or all((b >> 32 * i) & M32 != M32 for i in range(8))


def clip_b(op, b):
    """the nearest operand inside in_domain_b: every limb 0xFFFFFFFF lowered to 0xFFFFFFFE (the edge of the domain)"""
    if in_domain_b(op, b):
        return b
    return sum(min((b >> 32 * i) & M32, M32 - 1) << 32 * i for i in range(8))


def edge_classes(p, bound, rng):
    """the operand classes below `bound`"""
    v = {0, 1, (1 << 256) % p, p - 1, p - 2}
    for i in range(1, 8):
        v |= {(1 << 32 * i) - 1, (1 << 32 * i) + 1}
    # limb patterns over {0, 0xFFFFFFFF, p_i - 1, p_i + 1}: p with one limb replaced, uniform patterns, seeded mixtures
    pl = [(p >> 32 * i) & M32 for i in range(8)]
    choices = lambda i: (0, M32, (pl[i] - 1) & M32, (pl[i] + 1) & M32)
    join = lambda limbs: sum(x << 32 * i for i, x in enumerate(limbs))
    for i in range(8):
        for c in choices(i):
            v.add(join(pl[:i] + [c] + pl[i + 1:]))
    for k in range(4):
        v.add(join([choices(i)[k] for i in range(8)]))
    for _ in range(48):
        v.add(join([rng.choice(choices(i)) for i in range(8)]))
    # the top of the reduced range, [2^253, p)
    v |= {1 << 253, (1 << 253) + 1, p - 3} | {rng.randrange(1 << 253, p) for _ in range(4)}
    # unreduced left operands: [p, 2^254), [2^254, 2^255), 2^255 - 1, then [2^255, 2^256), 2^256 - 1
    v |= {p, p + 1, (1 << 254) - 1, 1 << 254, (1 << 255) - 2, (1 << 255) - 1, 1 << 255, (1 << 256) - 2, (1 << 256) - 1}
    v |= {rng.randrange(p, 1 << 254), rng.randrange(1 << 254, 1 << 255), rng.randrange(1 << 255, 1 << 256)}
    return sorted(x for x in v if x < bound)


def run_device(lib, field, op, a, b):
    n = len(a)
    pack = lambda xs: b"".join(x.to_bytes(32, "little") for x in xs)
    out = ctypes.create_string_buffer(32 * n)
    assert lib.h2v_selftest_field_vectors(0, field, OPS[op], n, pack(a), pack(b), out) == 0
    raw = out.raw
    return [int.from_bytes(raw[32 * i: 32 * i + 32], "little") for i in range(n)]


@pytest.mark.gpu
@pytest.mark.parametrize("op", list(OPS))
@pytest.mark.parametrize("fname", list(FIELDS))
def test_field_op_against_integers(pkg, fname, op):
    field, p = FIELDS[fname]
    rng = random.Random(f"field-vectors-{fname}-{op}")
    bound_a, bound_b = domain(op, p)
    ca = edge_classes(p, bound_a, rng)
    assert ca[0] == 0 and ca[-1] == bound_a - 1  # the classes reach both ends of the domain
    if op in BINARY:
        cb = sorted({clip_b(op, x) for x in edge_classes(p, bound_b, rng)})
        a = [x for x in ca for _ in cb]
        b = cb * len(ca)
    else:
        a, b = list(ca), [0] * len(ca)
    a += [rng.randrange(bound_a) for _ in range(RANDOM_PAIRS)]
    b += [clip_b(op, rng.randrange(bound_b)) if op in BINARY else 0 for _ in range(RANDOM_PAIRS)]
    got = run_device(pkg.load_library(), field, op, a, b)
    for x, y, g in zip(a, b, got):
        w = expected(op, p, x, y)
        assert g == w, f"{fname}.{op}({x:#x}, {y:#x}) = {g:#x}, expected {w:#x}"


def test_field_vectors_refuse_bad_arguments(built, pkg):
    """refused before any CUDA call: runs without a device"""
    lib = pkg.load_library()
    z = bytes(32)
    out = ctypes.create_string_buffer(32)
    assert lib.h2v_selftest_field_vectors(0, 2, 0, 1, z, z, out) == -1
    assert lib.h2v_selftest_field_vectors(0, 0, 13, 1, z, z, out) == -1
    assert lib.h2v_selftest_field_vectors(0, 1, -1, 1, z, z, out) == -1
    assert lib.h2v_selftest_field_vectors(0, 1, 0, 1, None, z, out) == -1


def test_expected_values_match_the_field_constants():
    """the reference formulas above against the Montgomery constants field.cuh hard-codes (R mod p, R^2 mod p)"""
    for _name, (_f, p) in FIELDS.items():
        R = 1 << 256
        assert expected("from_canonical", p, 1, 0) == R % p
        assert expected("mul", p, R % p, R % p) == R % p  # one * one = one
        assert expected("from_uniform", p, 0, 1) == R * R % p
        assert expected("inv", p, R % p, 0) == R % p
        for x in (2, p - 1, 12345):
            xm = x * R % p
            assert expected("mul", p, expected("inv", p, xm, 0), xm) == R % p
        # the right operands mul_any gets from from_canonical / from_uniform are inside its domain
        assert in_domain_b("mul_any", R * R % p) and in_domain_b("mul_any", R * R * R % p)
    assert not in_domain_b("mul_any", 0xFFFFFFFF) and in_domain_b("mul_any", clip_b("mul_any", (1 << 64) - 1))
    assert (1 << 256) % bn.R == 0x0E0A77C19A07DF2F666EA36F7879462E36FC76959F60CD29AC96341C4FFFFFFB
    assert (1 << 512) % bn.P == 0x06D89F71CAB8351F47AB1EFF0A417FF6B5E71911D44501FBF32CFC5B538AFA89

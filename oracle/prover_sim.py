"""Synthetic verifying keys and a trapdoor proof simulator (TEST INFRASTRUCTURE ONLY).

The reference ships no proofs or VKs and its prover (upstream halo2_proofs) is absent,
so accepting inputs are manufactured with the SRS trapdoor (SURVEY.md section 7):
every commitment gets a known discrete log, every evaluation is random, and the last
opening witness(es) are solved in the exponent from the verifier's own final equation
  SHPLONK  shplonk.rs:256-264:  s*c_h2 = sum_i scalar_i*dlog_i + u*c_h2
  GWC      gwc.rs:84-132:       s*w_i  = z_i*w_i + sum_j v^j c_ij - eval_batch_i   (per point)
The verifier does exactly the same work on these as on honest proofs.  LIMITATION: they
are self-consistent with the restated equations, so they cannot reveal a mis-transcribed
gate / permutation / lookup formula.

Shapes (SURVEY.md section 8):  "vm" = halo2_verifier/tests/vector_mul.rs:88-160 circuit,
"sh" = tests/shuffle.rs shape, "k18" = lookup+permutation-heavy synthetic, "mix" = small
shape exercising lookup + shuffle arguments, rotations and two phases together.
"""
import random

import bn254 as bn
from bn254 import R
from formats import COL_FIXED, COL_INSTANCE, ConstraintSystem, ParamsKZG, VerifyingKey
from verifier import OK, verify_proof

FIXTURE_SRS_SECRET = 0x1C59A59B6CFF4308740943526ADE1D8C09F71B337A67269CC89586BCDD6DFCBA


def make_params(k, s):
    return ParamsKZG(k, bn.G1_GEN, bn.G2_GEN, bn.g2_mul(bn.G2_GEN, s % R))


def _rand_poly(rng, n_vars, n_terms, max_deg, n_coeffs):
    terms = []
    for _ in range(n_terms):
        deg = rng.randint(1, max_deg)
        vars_ = {}
        for _ in range(deg):
            v = rng.randrange(n_vars)
            vars_[v] = vars_.get(v, 0) + 1
        terms.append((rng.randrange(n_coeffs), sorted(vars_.items())))
    return (n_vars, terms)


def make_vk(shape, k, seed=0):
    """Returns (vk, dlogs) with dlogs = {'fixed': [...], 'sigma': [...]}"""
    rng = random.Random(("vk", shape, k, seed).__repr__())
    cs = ConstraintSystem()
    if shape == "vm":
        cs.num_fixed_columns, cs.num_advice_columns, cs.num_instance_columns = 1, 3, 1
        cs.num_selectors, cs.num_challenges = 1, 0
        cs.advice_column_phase = [0, 0, 0]
        cs.num_advice_queries = [1, 1, 1]
        cs.advice_queries = [(0, 0, 0), (1, 0, 0), (2, 0, 0)]
        cs.instance_queries = [(0, 0)]
        cs.fixed_queries = [(0, 0)]
        cs.permutation_columns = [(0, COL_INSTANCE), (0, 0), (1, 0), (2, 0)]
        # s_mul * (lhs * rhs - out); variables: a0 a1 a2 | f0 | i0
        cs.gates = [(5, [(0, [(0, 1), (1, 1), (3, 1)]), (1, [(2, 1), (3, 1)])])]
        cs.coeff_vals = [1, R - 1]
        cs_degree = 3
    elif shape == "sh":
        cs.num_fixed_columns, cs.num_advice_columns, cs.num_instance_columns = 2, 9, 0
        cs.num_selectors, cs.num_challenges = 3, 2
        cs.advice_column_phase = [0] * 8 + [1]
        cs.challenge_phase = [0, 0]
        cs.num_advice_queries = [1] * 8 + [2]
        cs.advice_queries = [(c, 0, 0) for c in range(8)] + [(8, 1, 0), (8, 1, 1)]
        cs.fixed_queries = [(0, 0), (1, 0)]
        n_vars = 10 + 2 + 0 + 2
        cs.coeff_vals = [1, R - 1, rng.randrange(R)]
        cs.gates = [_rand_poly(rng, n_vars, 6, 4, 3) for _ in range(3)]
        cs_degree = 5
    elif shape == "mix":
        cs.num_fixed_columns, cs.num_advice_columns, cs.num_instance_columns = 3, 5, 2
        cs.num_selectors, cs.num_challenges = 2, 1
        cs.advice_column_phase = [0, 0, 0, 1, 1]
        cs.challenge_phase = [0]
        cs.num_advice_queries = [3, 1, 2, 1, 1]
        cs.advice_queries = [(0, 0, 0), (0, 0, 1), (0, 0, -1), (1, 0, 0), (2, 0, 0), (2, 0, 2), (3, 1, 0), (4, 1, 0)]
        cs.instance_queries = [(0, 0), (1, -1)]
        cs.fixed_queries = [(0, 0), (1, 1), (2, 0)]
        cs.permutation_columns = [(0, 0), (0, COL_INSTANCE), (2, COL_FIXED), (3, 1), (1, 0)]
        n_vars = 8 + 3 + 2 + 1
        cs.coeff_vals = [1, R - 1, rng.randrange(R), rng.randrange(R)]
        cs.gates = [_rand_poly(rng, n_vars, 5, 4, 4) for _ in range(4)]
        cs.lookups = [
            ([_rand_poly(rng, n_vars, 3, 2, 4) for _ in range(2)], [_rand_poly(rng, n_vars, 2, 1, 4) for _ in range(2)]),
            ([_rand_poly(rng, n_vars, 2, 2, 4)], [_rand_poly(rng, n_vars, 1, 1, 4)]),
        ]
        cs.shuffles = [([_rand_poly(rng, n_vars, 2, 2, 4)], [_rand_poly(rng, n_vars, 2, 2, 4)])]
        cs_degree = 5
    elif shape == "k18":
        cs.num_fixed_columns, cs.num_advice_columns, cs.num_instance_columns = 12, 64, 1
        cs.num_selectors, cs.num_challenges = 0, 0
        cs.advice_column_phase = [0] * 64
        cs.num_advice_queries = [3 if c < 20 else 1 for c in range(64)]
        cs.advice_queries = (
            [(c, 0, 0) for c in range(64)] + [(c, 0, 1) for c in range(20)] + [(c, 0, -1) for c in range(20)]
        )
        cs.instance_queries = [(0, 0)]
        cs.fixed_queries = [(c, 0) for c in range(12)]
        cs.permutation_columns = [(c, 0) for c in range(64)] + [(0, COL_FIXED), (0, COL_INSTANCE)]
        n_vars = 104 + 12 + 1
        cs.coeff_vals = [1, R - 1] + [rng.randrange(R) for _ in range(14)]
        cs.gates = [_rand_poly(rng, n_vars, 8, 5, 16) for _ in range(16)]
        cs.lookups = [
            ([_rand_poly(rng, n_vars, 3, 2, 16) for _ in range(2)], [_rand_poly(rng, n_vars, 2, 1, 16) for _ in range(2)])
            for _ in range(8)
        ]
        cs_degree = 5
    else:
        raise ValueError(shape)
    return vk_from_cs(k, cs, cs_degree, rng)


def vk_from_cs(k, cs, cs_degree, rng):
    """(vk, dlogs) of a constraint system: random fixed / sigma commitments with known discrete logs, random selectors
    and transcript_repr"""
    f_d = [rng.randrange(1, R) for _ in range(cs.num_fixed_columns)]
    s_d = [rng.randrange(1, R) for _ in range(len(cs.permutation_columns))]
    sel_bytes = ((1 << k) + 7) // 8
    vk = VerifyingKey(
        k=k,
        fixed_commitments=[bn.g1_mul_gen(d) for d in f_d],
        cs_degree=cs_degree,
        cs=cs,
        permutation_commitments=[bn.g1_mul_gen(d) for d in s_d],
        selectors=[bytes(rng.randrange(256) for _ in range(sel_bytes)) for _ in range(cs.num_selectors)],
        transcript_repr=rng.randrange(R),
    )
    return vk, {"fixed": f_d, "sigma": s_d}


def query_rotations(vk):
    """All query rotations in lib.rs:349-414 order (structure only)."""
    cs = vk.cs
    bf = cs.blinding_factors()
    chunk = vk.cs_degree - 2
    n_sets = -(-len(cs.permutation_columns) // chunk) if cs.permutation_columns else 0
    rots = [rot for _c, _p, rot in cs.advice_queries]
    rots += [0, 1] * n_sets + [-(bf + 1)] * max(0, n_sets - 1)
    rots += [0, 0, 0, -1, 1] * len(cs.lookups) + [0, 1] * len(cs.shuffles)
    rots += [rot for _c, rot in cs.fixed_queries] + [0] * len(vk.permutation_commitments) + [0, 0]
    return rots


def proof_layout(vk, multiopen="shplonk", m=1):
    """Item kinds ('P' compressed point / 'S' scalar) in transcript read order (lib.rs:86-253,
    then shplonk.rs:198-200 or gwc.rs:72-74); second value = index of the first multiopen item.
    m = circuit instances carried by the proof (`instances.len()`): the per-instance items repeat m times."""
    cs = vk.cs
    chunk = vk.cs_degree - 2
    n_sets = -(-len(cs.permutation_columns) // chunk) if cs.permutation_columns else 0
    items = []
    for phase in cs.phases():
        items += ["P"] * (m * sum(1 for p in cs.advice_column_phase if p == phase))
    items += ["P"] * (m * (2 * len(cs.lookups) + n_sets + len(cs.lookups) + len(cs.shuffles)) + 1)
    items += ["P"] * vk.quotient_poly_degree
    items += ["S"] * (m * len(cs.advice_queries) + len(cs.fixed_queries) + 1 + len(vk.permutation_commitments))
    items += ["S"] * (m * (3 * n_sets - 1 if n_sets else 0))
    items += ["S"] * (m * (5 * len(cs.lookups) + 2 * len(cs.shuffles)))
    first_multiopen = len(items)
    if multiopen == "shplonk":
        items += ["P", "P"]
    else:
        n = 1 << vk.k
        items += ["P"] * len({r % n for r in query_rotations(vk)})
    return items, first_multiopen


def random_instances(vk, rng, rows=10):
    return [[[rng.randrange(R) for _ in range(rows)] for _ in range(vk.cs.num_instance_columns)]]


def simulate_proof(params, vk, dlogs, s, instances, rng, multiopen="shplonk", hash_kind="blake2b"):
    """Returns accepting proof bytes for (params, vk, instances)."""
    items, first_mo = proof_layout(vk, multiopen, len(instances))
    slot_dlogs = []
    body = bytearray()
    for kind in items[:first_mo]:
        if kind == "P":
            c = rng.randrange(1, R)
            slot_dlogs.append(c)
            body += bn.g1_to_bytes(bn.g1_mul_gen(c))
        else:
            body += bn.fr_to_repr(rng.randrange(R))
    n_mo = len(items) - first_mo

    def dlog(ident):
        if ident[0] == "proof":
            return slot_dlogs[ident[1]]
        if ident[0] == "fixed":
            return dlogs["fixed"][ident[1]]
        if ident[0] == "sigma":
            return dlogs["sigma"][ident[1]]
        return 1 if ident == ("g",) else R - 1

    g_bytes = bn.g1_to_bytes(bn.G1_GEN)
    if multiopen == "shplonk":
        c_h1 = rng.randrange(1, R)
        slot_dlogs.append(c_h1)
        body += bn.g1_to_bytes(bn.g1_mul_gen(c_h1))
        res = verify_proof(params, vk, instances, bytes(body) + g_bytes, multiopen, hash_kind, False, False)
        assert res.status == OK, res.error
        h2_slot = len(slot_dlogs)
        acc = 0
        for sc, ident in zip(res.right.scalars, res.right.ids):
            if ident != ("proof", h2_slot):
                acc = (acc + sc * dlog(ident)) % R
        u = res.trace["shplonk_u"]
        c_h2 = acc * bn.fr_inv((s - u) % R) % R
        body += bn.g1_to_bytes(bn.g1_mul_gen(c_h2))
    else:
        res = verify_proof(params, vk, instances, bytes(body) + g_bytes * n_mo, multiopen, hash_kind, False, False)
        assert res.status == OK, res.error
        for z, batch, eval_batch in res.trace["gwc_per_point"]:
            acc = (-eval_batch) % R
            for sc, ident in zip(batch.scalars, batch.ids):
                acc = (acc + sc * dlog(ident)) % R
            w = acc * bn.fr_inv((s - z) % R) % R
            body += bn.g1_to_bytes(bn.g1_mul_gen(w))
    return bytes(body)


# ---------------------------------------------------------------- corruption injector
_NON_RESIDUE_X = None


def _offcurve_x():
    global _NON_RESIDUE_X
    if _NON_RESIDUE_X is None:
        x = 5
        while bn.fq_sqrt((x**3 + 3) % bn.P) is not None:
            x += 1
        _NON_RESIDUE_X = x
    return _NON_RESIDUE_X


CORRUPTIONS = (
    "eval_flip",  # -> ConstraintSystemFailure (the reference's own negative tests are of this kind)
    "point_swap",  # valid but wrong commitment -> ConstraintSystemFailure
    "scalar_ge_r",  # -> Transcript
    "point_offcurve",  # -> Transcript
    "point_x_ge_p",  # -> Transcript
    "point_identity",  # all-zero encoding -> Transcript
    "truncate_body",  # -> Transcript
    "opening_offcurve",  # multiopen point invalid -> Opening
    "truncate_opening",  # -> Opening
)


def corrupt(proof, vk, kind, rng, multiopen="shplonk", m=1):
    """Returns (corrupted proof, expected status); m = circuit instances carried by the proof."""
    from verifier import CONSTRAINT_SYSTEM_FAILURE, OPENING, TRANSCRIPT

    items, first_mo = proof_layout(vk, multiopen, m)
    b = bytearray(proof)
    pre_points = [i for i, k in enumerate(items[:first_mo]) if k == "P"]
    pre_scalars = [i for i, k in enumerate(items[:first_mo]) if k == "S"]
    mo = list(range(first_mo, len(items)))
    if kind == "eval_flip":
        i = rng.choice(pre_scalars)
        b[32 * i] ^= 1
        v = int.from_bytes(b[32 * i : 32 * i + 32], "little")
        if v >= R:  # keep the encoding canonical
            b[32 * i] ^= 3
        return bytes(b), CONSTRAINT_SYSTEM_FAILURE
    if kind == "point_swap":
        i = rng.choice(pre_points)
        b[32 * i : 32 * i + 32] = bn.g1_to_bytes(bn.g1_mul_gen(rng.randrange(1, R)))
        return bytes(b), CONSTRAINT_SYSTEM_FAILURE
    if kind == "scalar_ge_r":
        i = rng.choice(pre_scalars)
        b[32 * i : 32 * i + 32] = (R + rng.randrange(1 << 64)).to_bytes(32, "little")
        return bytes(b), TRANSCRIPT
    if kind == "point_offcurve":
        i = rng.choice(pre_points)
        b[32 * i : 32 * i + 32] = _offcurve_x().to_bytes(32, "little")
        return bytes(b), TRANSCRIPT
    if kind == "point_x_ge_p":
        i = rng.choice(pre_points)
        b[32 * i : 32 * i + 32] = (bn.P + 1).to_bytes(32, "little")
        return bytes(b), TRANSCRIPT
    if kind == "point_identity":
        i = rng.choice(pre_points)
        b[32 * i : 32 * i + 32] = bytes(32)
        return bytes(b), TRANSCRIPT
    if kind == "truncate_body":
        cut = rng.randrange(1, 32 * first_mo)
        return bytes(b[:cut]), TRANSCRIPT
    if kind == "opening_offcurve":
        i = rng.choice(mo)
        b[32 * i : 32 * i + 32] = _offcurve_x().to_bytes(32, "little")
        return bytes(b), OPENING
    if kind == "truncate_opening":
        cut = rng.randrange(32 * first_mo, 32 * len(items))
        return bytes(b[:cut]), OPENING
    raise ValueError(kind)

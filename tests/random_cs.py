"""Seeded random constraint systems and the VKs at the plan's build limits (oracle-side generation: TEST INFRASTRUCTURE).

random_vk varies everything the plan compiler (csrc/plan_build.cpp) derives from a VK: the transcript schedule (phases,
challenges, lookups, shuffles, permutation chunks), rotation dedup modulo n, SHPLONK rotation sets, GWC points, instance
offsets and expression terms.  limit_vk builds a VK exactly at one of the fixed-size arrays of the device code (plan.h), or
one past it."""
import random

from bn254 import R
from formats import COL_FIXED, COL_INSTANCE, ConstraintSystem
import prover_sim as sim


def _finish(rng, k, cs, cs_degree, n_gates, lookups=(), shuffles=()):
    """coefficients, gates over every polynomial variable (advice queries | fixed | instance | challenges), lookups and
    shuffles given as lists of expression-pair counts"""
    n_vars = len(cs.advice_queries) + cs.num_fixed_columns + cs.num_instance_columns + cs.num_challenges
    cs.coeff_vals = [1, R - 1] + [rng.randrange(R) for _ in range(rng.randint(1, 3))]
    nc = len(cs.coeff_vals)
    cs.gates = [sim._rand_poly(rng, n_vars, rng.randint(1, 5), cs_degree - 1, nc) for _ in range(n_gates)]
    cs.lookups = [([sim._rand_poly(rng, n_vars, rng.randint(1, 3), 2, nc) for _ in range(p)],
                   [sim._rand_poly(rng, n_vars, rng.randint(1, 2), 1, nc) for _ in range(p)]) for p in lookups]
    cs.shuffles = [([sim._rand_poly(rng, n_vars, rng.randint(1, 3), 2, nc) for _ in range(p)],
                    [sim._rand_poly(rng, n_vars, rng.randint(1, 3), 2, nc) for _ in range(p)]) for p in shuffles]
    return sim.vk_from_cs(k, cs, cs_degree, rng)


def random_vk(rng, k):
    """(vk, dlogs) of a random constraint system at 2^k rows that the reference's `read` accepts and prover_sim can prove"""
    n = 1 << k
    cs = ConstraintSystem()
    n_adv, last_phase = rng.randint(1, 6), rng.randint(0, 2)
    cs.advice_column_phase = [rng.randint(0, last_phase) for _ in range(n_adv)]
    cs.advice_column_phase[rng.randrange(n_adv)] = last_phase  # earlier phases may be empty
    cs.num_advice_columns, cs.num_instance_columns, cs.num_fixed_columns = n_adv, rng.randint(0, 3), rng.randint(1, 4)
    cs.num_selectors, cs.num_challenges = rng.randint(0, 2), rng.randint(0, 3)
    cs.challenge_phase = [rng.randint(0, last_phase) for _ in range(cs.num_challenges)]
    cs_degree = rng.randint(3, 9)

    # permutation: a column count on a multiple of the chunk length (cs_degree - 2), one below it, one above it, or none
    chunk = cs_degree - 2
    pool = [(c, cs.advice_column_phase[c]) for c in range(n_adv)] + [(i, COL_INSTANCE) for i in range(cs.num_instance_columns)] + \
           [(f, COL_FIXED) for f in range(cs.num_fixed_columns)]
    delta = rng.choice((None, 0, -1, 1))
    counts = [] if delta is None else [c for c in range(1, len(pool) + 1) if c - delta > 0 and (c - delta) % chunk == 0]
    cs.permutation_columns = rng.sample(pool, rng.choice(counts)) if counts else []
    in_perm = set(cs.permutation_columns)

    # advice queries: distinct integer rotations per column, some equal mod n, and -(blinding_factors + 1) among them
    cs.num_advice_queries = [rng.randint(1, 5) for _ in range(n_adv)]
    bf = cs.blinding_factors()
    rots = [0, 1, -1, 2, -2, 3, -5, 7, n // 2, n - 1, -(n - 1), -(bf + 1)]
    queries = []
    for c in range(n_adv):
        rs = rng.sample(rots, cs.num_advice_queries[c])
        if (c, cs.advice_column_phase[c]) in in_perm and 0 not in rs:
            rs[0] = 0  # the permutation argument reads every column at Rotation::cur()
        queries += [(c, cs.advice_column_phase[c], r) for r in rs]
    rng.shuffle(queries)
    cs.advice_queries = queries
    cs.instance_queries = [(i, 0 if (i, COL_INSTANCE) in in_perm else rng.choice((-1, 0, 1, 2))) for i in range(cs.num_instance_columns)]
    cs.fixed_queries = [(f, 0 if (f, COL_FIXED) in in_perm else rng.choice((-1, 0, 1, 2))) for f in range(cs.num_fixed_columns)]

    lookups = [rng.randint(1, 3) for _ in range(rng.randint(0, 2))]
    shuffles = [rng.randint(1, 2) for _ in range(rng.randint(0, 2))]
    vk, dl = _finish(rng, k, cs, cs_degree, rng.randint(1, 3), lookups, shuffles)
    if cs.num_challenges and cs.lookups:  # a challenge as a variable of a lookup input
        ch_var = len(cs.advice_queries) + cs.num_fixed_columns + cs.num_instance_columns + rng.randrange(cs.num_challenges)
        nv, terms = cs.lookups[0][0][0]
        cs.lookups[0][0][0] = (nv, terms + [(0, [(ch_var, 1)])])
    return vk, dl


def usable_rows(vk):
    """rows of a column a circuit can assign: n - (blinding_factors + 1)"""
    return vk.n - (vk.cs.blinding_factors() + 1)


# the fixed-size arrays of the per-proof stages (csrc/plan.h) and the plan compiler's message one past each
LIMIT_ERRORS = {
    "set_points": "rotation set too large for this build",     # H2V_MAX_SET_POINTS = 8: basis[] of a SHPLONK set
    "rot": "too many distinct rotations for this build",        # H2V_MAX_ROT = 32: um[]
    "inst_q": "too many instance queries for this build",       # H2V_MAX_INST_Q = 16: ie[], instance columns x m
    "levals": "too many blinding factors for this build",       # H2V_MAX_LEVALS = 64: pre[], blinding_factors + 2
}


def limit_vk(which, at_limit, m=1):
    """(vk, dlogs) exactly at one build limit (at_limit) or one past it; m = circuit instances per proof (inst_q only)"""
    rng = random.Random(repr(("limit", which, at_limit, m)))
    cs = ConstraintSystem()
    cs.num_fixed_columns, cs.fixed_queries = 1, [(0, 0)]
    n_inst = 0
    if which == "set_points":  # one commitment opened at 8 (9) points: one SHPLONK set of that size
        k, cols = 5, [[0, 1, -1, 2, -2, 3, -3, 4] + ([5] if not at_limit else [])]
    elif which == "rot":  # 32 (33) distinct points, at most 8 per commitment
        k, cols = 7, [list(range(8 * c, 8 * c + 8)) for c in range(4)] + ([[32]] if not at_limit else [])
    elif which == "inst_q":  # instance columns x m = 16 (one more column past it)
        k, cols, n_inst = 5, [[0]], 16 // m + (0 if at_limit else 1)
    elif which == "levals":  # 60 (61) queries of one column: blinding_factors + 2 = 64 (65), on 4 (5) points mod n = 16
        k, cols = 4, [[r + 16 * t for r in (0, 1, -1, 2) for t in range(15)] + ([3] if not at_limit else [])]
    else:
        raise ValueError(which)
    cs.num_advice_columns = len(cols)
    cs.advice_column_phase = [0] * len(cols)
    cs.num_advice_queries = [len(c) for c in cols]
    cs.advice_queries = [(c, 0, r) for c, rs in enumerate(cols) for r in rs]
    cs.num_instance_columns = n_inst
    cs.instance_queries = [(i, 0) for i in range(n_inst)]
    return _finish(rng, k, cs, 3, 2)

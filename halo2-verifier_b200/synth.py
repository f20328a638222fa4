"""Synthetic workloads for benchmarks: VK bytes of the named circuit shapes and a GPU-assisted
trapdoor proof synthesiser.

The reference ships no proofs and its prover (upstream halo2_proofs) is not available offline, so
benchmark inputs are manufactured (SURVEY.md section 7): every commitment is [c]G with a known c,
every evaluation is random, and the last SHPLONK opening witness h2 is solved in the exponent from
the verifier's final equation (reference shplonk.rs:256-264)

        s * c_h2 = sum_b scalar_b * dlog_b + u * c_h2          (u is the scalar of h2 itself)

The per-base scalars come from the device (the `msm_scalars` parity hook of the C ABI) in a first
pass over proofs that carry a placeholder h2; h2 is the last item of the transcript, so nothing
else depends on it.  The verifier then does exactly the work it does on honest proofs.  This module
is a workload generator, not a verifier: correctness of the device path is established separately
against the CPU oracle in tests/.

VK bytes follow what the reference's `VerifyingKey::read` expects (plonk/vk.rs:76-115,274-365).
"""
import random
import struct

P = 0x30644E72E131A029B85045B68181585D97816A916871CA8D3C208C16D87CFD47
R = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001
G1 = (1, 2)
# BN254 G2 generator and its negation are public constants; [s]G2 needs G2 arithmetic (below)
G2 = ((0x1800DEEF121F1E76426A00665E5C4479674322D4F75EDADD46DEBD5CD992F6ED, 0x198E9393920D483A7260BFB731FB5D25F1AA493335A9E71297E485B7AEF312C2),
      (0x12C85EA5DB8C6DEB4AAB71808DCB408FE3D1E7690C43D37B4CE6CC0166FA7DAA, 0x090689D0585FF075EC9E99AD690C3395BC4B313370B38EF355ACDADCD122975B))
MONT = 1 << 256


# ---------------------------------------------------------------- minimal group arithmetic (host, big ints)
def g1_add(a, b):
    if a is None:
        return b
    if b is None:
        return a
    x1, y1 = a
    x2, y2 = b
    if x1 == x2:
        if (y1 + y2) % P == 0:
            return None
        lam = 3 * x1 * x1 * pow(2 * y1, -1, P) % P
    else:
        lam = (y2 - y1) * pow(x2 - x1, -1, P) % P
    x3 = (lam * lam - x1 - x2) % P
    return (x3, (lam * (x1 - x3) - y1) % P)


class _Table:
    """8-bit fixed-base windows of G: [k]G in <= 32 affine additions."""

    def __init__(self):
        self.rows = []
        b = G1
        for _ in range(32):
            row, acc = [None], None
            for _ in range(255):
                acc = g1_add(acc, b)
                row.append(acc)
            self.rows.append(row)
            b = g1_add(acc, b)

    def mul(self, k):
        k %= R
        acc, i = None, 0
        while k:
            if k & 0xFF:
                acc = g1_add(acc, self.rows[i][k & 0xFF])
            k >>= 8
            i += 1
        return acc


_TABLE = None


def g1_mul_gen(k):
    global _TABLE
    if _TABLE is None:
        _TABLE = _Table()
    return _TABLE.mul(k)


def _f2_mul(a, b):
    return ((a[0] * b[0] - a[1] * b[1]) % P, (a[0] * b[1] + a[1] * b[0]) % P)


def _f2_inv(a):
    d = pow(a[0] * a[0] + a[1] * a[1], -1, P)
    return (a[0] * d % P, -a[1] * d % P)


def _g2_add(a, b):
    if a is None:
        return b
    if b is None:
        return a
    (x1, y1), (x2, y2) = a, b
    if x1 == x2:
        if ((y1[0] + y2[0]) % P, (y1[1] + y2[1]) % P) == (0, 0):
            return None
        x1s = _f2_mul(x1, x1)
        lam = _f2_mul((3 * x1s[0] % P, 3 * x1s[1] % P), _f2_inv((2 * y1[0] % P, 2 * y1[1] % P)))
    else:
        lam = _f2_mul(((y2[0] - y1[0]) % P, (y2[1] - y1[1]) % P), _f2_inv(((x2[0] - x1[0]) % P, (x2[1] - x1[1]) % P)))
    l2 = _f2_mul(lam, lam)
    x3 = ((l2[0] - x1[0] - x2[0]) % P, (l2[1] - x1[1] - x2[1]) % P)
    t = _f2_mul(lam, ((x1[0] - x3[0]) % P, (x1[1] - x3[1]) % P))
    return (x3, ((t[0] - y1[0]) % P, (t[1] - y1[1]) % P))


def g2_mul_gen(k):
    acc, add = None, G2
    k %= R
    while k:
        if k & 1:
            acc = _g2_add(acc, add)
        add = _g2_add(add, add)
        k >>= 1
    return acc


def g1_compress(pt):
    x, y = pt
    b = bytearray(x.to_bytes(32, "little"))
    if y & 1:
        b[31] |= 0x80
    return bytes(b)


def g1_raw(pt):
    return (pt[0] * MONT % P).to_bytes(32, "little") + (pt[1] * MONT % P).to_bytes(32, "little")


def params_bytes_raw(k, s):
    """ParamsKZG in RawBytes form: u32le k | G1 g | G2 g2 | G2 s_g2 (kzg/commitment.rs:142-152)."""
    sg2 = g2_mul_gen(s)
    raw2 = lambda q: b"".join((v * MONT % P).to_bytes(32, "little") for v in (q[0][0], q[0][1], q[1][0], q[1][1]))
    return struct.pack("<I", k) + g1_raw(G1) + raw2(G2) + raw2(sg2)


# ---------------------------------------------------------------- VK bytes (RawBytes) of the named shapes
def _poly(num_vars, terms):
    out = struct.pack(">II", num_vars, len(terms))
    for coeff, vars_ in terms:
        out += struct.pack(">HI", coeff, len(vars_))
        for var, pw in vars_:
            out += struct.pack(">II", var, pw)
    return out


def _rand_poly(rng, n_vars, n_terms, max_deg, n_coeffs):
    terms = []
    for _ in range(n_terms):
        vars_ = {}
        for _ in range(rng.randint(1, max_deg)):
            v = rng.randrange(n_vars)
            vars_[v] = vars_.get(v, 0) + 1
        terms.append((rng.randrange(n_coeffs), sorted(vars_.items())))
    return _poly(n_vars, terms)


def make_vk_bytes(shape, k, seed=0):
    """Returns (vk bytes in RawBytes format, dlogs of the shared bases [fixed..., sigma..., G]).
    "vm": the circuit of reference halo2_verifier/tests/vector_mul.rs:88-160 (3 advice, 1 instance,
    1 fixed selector column, one degree-3 gate, permutation over 4 columns).
    "k18": lookup+permutation-heavy synthetic shape of BASELINE.json config 4 (64 advice columns,
    104 advice queries, 12 fixed, 16 gates of degree <= 5, 8 lookups, permutation over 66 columns)."""
    rng = random.Random(repr(("bench-vk", shape, k, seed)))
    fr = lambda v: (v * MONT % R).to_bytes(32, "little")
    if shape == "vm":
        n_fixed, n_adv, n_inst, n_sel, n_ch = 1, 3, 1, 1, 0
        adv_phase, ch_phase, n_adv_q = [0, 0, 0], [], [1, 1, 1]
        adv_q = [(0, 0, 0), (1, 0, 0), (2, 0, 0)]
        inst_q, fixed_q = [(0, 0)], [(0, 0)]
        perm = [(0, 254), (0, 0), (1, 0), (2, 0)]
        gates = [_poly(5, [(0, [(0, 1), (1, 1), (3, 1)]), (1, [(2, 1), (3, 1)])])]
        lookups, coeffs, cs_degree = [], [1, R - 1], 3
    elif shape == "k18":
        n_fixed, n_adv, n_inst, n_sel, n_ch = 12, 64, 1, 0, 0
        adv_phase, ch_phase = [0] * 64, []
        n_adv_q = [3 if c < 20 else 1 for c in range(64)]
        adv_q = [(c, 0, 0) for c in range(64)] + [(c, 0, 1) for c in range(20)] + [(c, 0, -1) for c in range(20)]
        inst_q, fixed_q = [(0, 0)], [(c, 0) for c in range(12)]
        perm = [(c, 0) for c in range(64)] + [(0, 255), (0, 254)]
        nv = 104 + 12 + 1
        coeffs = [1, R - 1] + [rng.randrange(R) for _ in range(14)]
        gates = [_rand_poly(rng, nv, 8, 5, 16) for _ in range(16)]
        lookups = [([_rand_poly(rng, nv, 3, 2, 16) for _ in range(2)], [_rand_poly(rng, nv, 2, 1, 16) for _ in range(2)]) for _ in range(8)]
        cs_degree = 5
    else:
        raise ValueError(shape)
    f_d = [rng.randrange(1, R) for _ in range(n_fixed)]
    s_d = [rng.randrange(1, R) for _ in range(len(perm))]
    out = struct.pack(">II", k, n_fixed) + b"".join(g1_raw(g1_mul_gen(d)) for d in f_d)
    out += struct.pack(">I", cs_degree)
    out += struct.pack(">9I", n_fixed, n_adv, n_inst, n_sel, n_ch, len(gates), len(lookups), 0, len(coeffs))
    out += bytes(adv_phase) + bytes(ch_phase) + b"".join(struct.pack(">I", c) for c in n_adv_q)
    out += b"".join(struct.pack(">IBi", *q) for q in adv_q)
    out += b"".join(struct.pack(">Ii", *q) for q in inst_q) + b"".join(struct.pack(">Ii", *q) for q in fixed_q)
    out += struct.pack(">I", len(perm)) + b"".join(struct.pack(">IB", *c) for c in perm)
    out += b"".join(gates)
    for ins, tabs in lookups:
        out += struct.pack(">I", len(ins)) + b"".join(a + b for a, b in zip(ins, tabs))
    out += b"".join(fr(c) for c in coeffs)
    out += b"".join(g1_raw(g1_mul_gen(d)) for d in s_d)
    out += bytes(n_sel * (((1 << k) + 7) // 8))
    out += fr(rng.randrange(R))
    return out, f_d + s_d + [1]


def _layout(bv):
    """'P' / 'S' item kinds of a proof in transcript order, from the context's shape only:
    points and scalars are each contiguous runs in the C ABI's slot order, but interleaved in the
    proof; the multi-open points are the last n_mo items, every scalar precedes them, and the
    non-multi-open points precede the scalars (reference lib.rs:86-253)."""
    return ["P"] * (bv.n_points - bv.n_mo) + ["S"] * bv.n_scalars + ["P"] * bv.n_mo


def synthesize_shplonk_batch(bv, shared_dlogs, s, n, seed, rows=10, instances_of=None):
    """n accepting SHPLONK proofs + public inputs for the context `bv` (a BatchVerifier, plain: it parses the placeholders).
    instances_of(j, rng) (optional) gives proof j's instances[column][row] as 32-byte strings instead of random ones.
    Returns (list of proof bytes, list of instances[column][row] as 32-byte strings)."""
    assert bv.n_mo == 2, "SHPLONK contexts only"
    rng = random.Random(repr(("bench-batch", seed, n)))
    walk = [(d, g1_mul_gen(d)) for d in (rng.randrange(1, R) for _ in range(64))]  # known-dlog steps
    cur_d = rng.randrange(1, R)
    cur = g1_mul_gen(cur_d)
    g_c = g1_compress(G1)
    proofs, dlogs, instances = [], [], []
    n_pre = bv.n_points - 2
    for _ in range(n):
        body, dl = bytearray(), []
        for _i in range(n_pre + 1):  # commitments + h1: a random walk over known discrete logs
            d, pt = walk[rng.randrange(64)]
            cur, cur_d = g1_add(cur, pt), (cur_d + d) % R
            if cur is None:
                cur_d = rng.randrange(1, R)
                cur = g1_mul_gen(cur_d)
            dl.append(cur_d)
            if _i == n_pre:
                h1 = g1_compress(cur)
            else:
                body += g1_compress(cur)
        body += b"".join(rng.randrange(R).to_bytes(32, "little") for _ in range(bv.n_scalars))
        proofs.append(bytes(body) + h1 + g_c)
        dlogs.append(dl)
        instances.append(instances_of(len(instances), rng) if instances_of else
                         [[rng.randrange(R).to_bytes(32, "little") for _ in range(rows)] for _ in range(bv.n_inst_cols)])
    res = bv.verify_batch(proofs, instances, want_scalars=True)
    nb, P_, Sh = bv.n_bases, bv.n_points, bv.n_shared
    out = []
    for j in range(n):
        assert res.status[j] in (0, 4), f"placeholder proof {j} was not parsed (status {res.status[j]})"
        sc = [int.from_bytes(res.msm_scalars[32 * (j * nb + b): 32 * (j * nb + b + 1)], "little") for b in range(P_ + Sh)]
        acc = sum(sc[b] * dlogs[j][b] for b in range(P_ - 1)) + sum(sc[P_ + b] * shared_dlogs[b] for b in range(Sh))
        u = sc[P_ - 1]
        c_h2 = acc % R * pow((s - u) % R, -1, R) % R
        out.append(proofs[j][:-32] + g1_compress(g1_mul_gen(c_h2)))
    return out, instances

"""Pins the oracle's arithmetic against the reference's only binary fixture (kzg_bn254_8.srs, via the
committed extract tests/golden/srs_kat.json) and against standard hash KATs; then checks the oracle's
verifier on simulated proofs of every shape (accept / every rejection class)."""
import hashlib
import json
import os
import random

import pytest

import bn254 as bn
import formats as F
import prover_sim as sim
import transcript as T
import verifier as orc
from workloads import setup

HERE = os.path.dirname(os.path.abspath(__file__))
KAT = json.load(open(os.path.join(HERE, "golden", "srs_kat.json")))
S = sim.FIXTURE_SRS_SECRET


def _g1(hexs):
    ok, pt = bn.g1_read_raw(bytes.fromhex(hexs))
    assert ok
    return pt


def test_srs_fixture_extract_matches_live_file():
    # the fixture file as the reference's gen_srs writes it (tests/golden/make_srs_fixture.py)
    raw = open(os.path.join(HERE, "golden", "kzg_bn254_8.srs"), "rb").read()
    assert len(raw) == 33028
    assert raw[:4].hex() == KAT["k_le"] and raw[4:68].hex() == KAT["g"]["0"]
    assert raw[-128:].hex() == KAT["s_g2"] and raw[-256:-128].hex() == KAT["g2"]
    off_l = 4 + 256 * 64
    for i, v in KAT["g"].items():
        assert raw[4 + 64 * int(i): 4 + 64 * (int(i) + 1)].hex() == v
    for i, v in KAT["g_lagrange"].items():
        assert raw[off_l + 64 * int(i): off_l + 64 * (int(i) + 1)].hex() == v
    params = F.params_from_srs_fixture(raw)
    assert params.k == 8 and params.g == bn.G1_GEN and params.s_g2 == bn.g2_mul(bn.G2_GEN, S)


def test_srs_secret_is_chacha20_zero_key():
    # Fr::random = 512-bit LE reduction of RNG output; ChaCha20 block 0 with zero key / nonce
    def chacha_block0():
        st = [0x61707865, 0x3320646E, 0x79622D32, 0x6B206574] + [0] * 12
        w = list(st)
        rot = lambda v, n: ((v << n) | (v >> (32 - n))) & 0xFFFFFFFF

        def qr(a, b, c, d):
            w[a] = (w[a] + w[b]) & 0xFFFFFFFF; w[d] = rot(w[d] ^ w[a], 16)
            w[c] = (w[c] + w[d]) & 0xFFFFFFFF; w[b] = rot(w[b] ^ w[c], 12)
            w[a] = (w[a] + w[b]) & 0xFFFFFFFF; w[d] = rot(w[d] ^ w[a], 8)
            w[c] = (w[c] + w[d]) & 0xFFFFFFFF; w[b] = rot(w[b] ^ w[c], 7)

        for _ in range(10):
            qr(0, 4, 8, 12); qr(1, 5, 9, 13); qr(2, 6, 10, 14); qr(3, 7, 11, 15)
            qr(0, 5, 10, 15); qr(1, 6, 11, 12); qr(2, 7, 8, 13); qr(3, 4, 9, 14)
        return b"".join(((a + b) & 0xFFFFFFFF).to_bytes(4, "little") for a, b in zip(w, st))

    assert bn.fr_from_uniform_bytes(chacha_block0()) == S


def test_g1_g2_field_layout_against_fixture():
    assert int.from_bytes(bytes.fromhex(KAT["k_le"]), "little") == 8
    assert _g1(KAT["g"]["0"]) == bn.G1_GEN
    for i in (1, 2, 3, 255):
        assert _g1(KAT["g"][str(i)]) == bn.g1_mul(bn.G1_GEN, pow(S, i, bn.R))
    # g_lagrange[i] = [L_i(s)]G with omega = ROOT_OF_UNITY^(2^(28-8)): pins ROOT_OF_UNITY (hence generator 7, DELTA)
    n, omega = 256, pow(bn.FR_ROOT_OF_UNITY, 1 << 20, bn.R)
    assert pow(omega, n, bn.R) == 1 and pow(omega, n // 2, bn.R) != 1
    for i in (0, 1, 2, 255):
        wi = pow(omega, i, bn.R)
        li = (pow(S, n, bn.R) - 1) * bn.fr_inv(n) % bn.R * wi % bn.R * bn.fr_inv((S - wi) % bn.R) % bn.R
        assert _g1(KAT["g_lagrange"][str(i)]) == bn.g1_mul(bn.G1_GEN, li)
    ok, g2 = bn.g2_read_raw(bytes.fromhex(KAT["g2"]))
    ok2, s_g2 = bn.g2_read_raw(bytes.fromhex(KAT["s_g2"]))
    assert ok and ok2 and g2 == bn.G2_GEN and s_g2 == bn.g2_mul(bn.G2_GEN, S)


def test_pairing_against_fixture_and_bilinearity():
    _, s_g2 = bn.g2_read_raw(bytes.fromhex(KAT["s_g2"]))
    a = 0x1234567890ABCDEF
    assert bn.pairing_check([(bn.g1_mul_gen(a), s_g2), (bn.g1_mul_gen(a * S % bn.R), bn.g2_neg(bn.G2_GEN))])
    assert not bn.pairing_check([(bn.g1_mul_gen(a), s_g2), (bn.g1_mul_gen((a * S + 1) % bn.R), bn.g2_neg(bn.G2_GEN))])
    e = bn.pairing(bn.G1_GEN, bn.G2_GEN)
    assert bn.pairing(bn.g1_mul_gen(5), bn.g2_mul(bn.G2_GEN, 7)) == bn.f12_pow(e, 35) != bn.F12_ONE
    assert bn.f12_pow(e, bn.R) == bn.F12_ONE


def test_hash_kats():
    assert T.keccak256(b"").hex() == "c5d2460186f7233c927e7db2dcc703c0e500b653ca82273b7bfad8045d85a470"
    assert T.keccak256(b"abc").hex() == "4e03657aea45a94fc7d47ba826c8d667c0d1e6e33a64a036ec44f58fa12d6c45"
    t = T.TranscriptRead(b"", "blake2b")
    t.state.update(b"\x00")
    assert t.state.copy().digest().hex().startswith("c8ed8d1468d8f56b")  # SURVEY.md 5.1
    assert hashlib.blake2b(b"\x00", digest_size=64, person=b"Halo2-Transcript").digest() == t.state.digest()


def test_constants():
    assert bn.FR_ROOT_OF_UNITY == pow(7, (bn.R - 1) >> 28, bn.R)
    assert bn.FR_DELTA == pow(7, 1 << 28, bn.R)
    assert (bn.P**12 - 1) % bn.R == 0 and (bn.P**6 - 1) % bn.R != 0
    assert bn.fq_sqrt(3) is None  # x = 0 never decompresses


@pytest.mark.parametrize("shape,k", [("vm", 8), ("sh", 8), ("mix", 6)])
@pytest.mark.parametrize("mo", ["shplonk", "gwc"])
@pytest.mark.parametrize("hk", ["blake2b", "keccak"])
def test_oracle_accepts_and_rejects(shape, k, mo, hk):
    params, vk, dl, s = setup(shape, k)
    rng = random.Random(f"{shape}{k}{mo}{hk}")
    for fmt in (F.PROCESSED, F.RAW_BYTES):
        vb = vk.to_bytes(fmt)
        assert F.VerifyingKey.from_bytes(vb, fmt).to_bytes(fmt) == vb
    pb = params.to_bytes()
    assert len(pb) == 164 and F.ParamsKZG.from_bytes(pb).to_bytes() == pb
    inst = sim.random_instances(vk, rng, 10)
    proof = sim.simulate_proof(params, vk, dl, s, inst, rng, mo, hk)
    items, _ = sim.proof_layout(vk, mo)
    assert len(proof) == 32 * len(items)
    assert orc.verify_proof(params, vk, inst, proof, mo, hk).status == orc.OK
    if hk == "blake2b":
        for kind in sim.CORRUPTIONS:
            bad, exp = sim.corrupt(proof, vk, kind, rng, mo)
            assert orc.verify_proof(params, vk, inst, bad, mo, hk, check_pairing=exp == 4).status == exp, kind
    if vk.cs.num_instance_columns:  # the reference's own negative test: bump a public input (vector_mul.rs:327-330)
        inst2 = [[list(c) for c in inst[0]]]
        inst2[0][0][0] = (inst2[0][0][0] + 1) % bn.R
        assert orc.verify_proof(params, vk, inst2, proof, mo, hk).status == orc.CONSTRAINT_SYSTEM_FAILURE
        assert orc.verify_proof(params, vk, [inst[0][:-1]], proof, mo, hk).status == orc.INVALID_INSTANCES


def test_vm_proof_size_matches_survey():
    _p, vk, _d, _s = setup("vm", 8)
    assert 32 * len(sim.proof_layout(vk, "shplonk")[0]) == 1024  # SURVEY.md Appendix B
    assert 32 * len(sim.proof_layout(vk, "gwc")[0]) == 1056


def test_rlc_convention():
    rs = [3, 5, 7, 11]
    assert orc.rlc_coefficients(rs) == [5 * 7 * 11, 7 * 11, 11, 1]  # c_j = prod_{i>j} r_i (strategy.rs:125-136)


def test_golden_vectors_reproduce():
    for fn in sorted(os.listdir(os.path.join(HERE, "golden"))):
        if not fn.endswith(".json") or fn == "srs_kat.json":
            continue
        g = json.load(open(os.path.join(HERE, "golden", fn)))
        params = F.ParamsKZG.from_bytes(bytes.fromhex(g["params"]))
        vk = F.VerifyingKey.from_bytes(bytes.fromhex(g["vk"]), g["vk_format"])
        for e in g["proofs"]:
            if "circuit_instances" in g:
                inst = [[[int(v, 16) for v in col] for col in ci] for ci in e["instances"]]
            else:
                inst = [[[int(v, 16) for v in col] for col in e["instances"]]]
            res = orc.verify_proof(params, vk, inst, bytes.fromhex(e["proof"]), g["multiopen"], g["hash"])
            assert res.status == e["status"] and [hex(c) for c in res.challenges] == e["challenges"], fn

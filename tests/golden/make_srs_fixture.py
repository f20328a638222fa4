"""Writes tests/golden/kzg_bn254_8.srs, the reference's SRS fixture halo2_verifier/params/kzg_bn254_8.srs, rebuilt the
way the reference's gen_srs builds it when the file is absent (tests/helpers.rs:87-105): ParamsKZG::setup(8, rng) with
ChaCha20Rng::from_seed(Default::default()), whose secret is prover_sim.FIXTURE_SRS_SECRET (test_oracle_kat.py
checks that).  Layout (upstream PSE RawBytes): u32le k | 2^k G1 g[i] = [s^i]G | 2^k G1 g_lagrange[i] = [L_i(s)]G |
G2 g2 | G2 s_g2, coordinates in Montgomery form.  Every point is a function of s alone, so the rebuilt bytes equal the
reference's; the script checks them against the extract srs_kat.json taken from the reference's own file before it
writes.  Run:  python tests/golden/make_srs_fixture.py"""
import json, os, struct, sys
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", "..", "oracle"))
import bn254 as bn, prover_sim as sim

k, s = 8, sim.FIXTURE_SRS_SECRET
n = 1 << k
omega = pow(bn.FR_ROOT_OF_UNITY, 1 << (28 - k), bn.R)
g = [bn.g1_mul_gen(pow(s, i, bn.R)) for i in range(n)]
zn = (pow(s, n, bn.R) - 1) * bn.fr_inv(n) % bn.R  # L_i(s) = (s^n - 1) / n * w^i / (s - w^i)
lag = [bn.g1_mul_gen(zn * pow(omega, i, bn.R) % bn.R * bn.fr_inv((s - pow(omega, i, bn.R)) % bn.R)) for i in range(n)]
raw = (struct.pack("<I", k) + b"".join(bn.g1_write_raw(p) for p in g + lag)
       + bn.g2_write_raw(bn.G2_GEN) + bn.g2_write_raw(bn.g2_mul(bn.G2_GEN, s)))
kat = json.load(open(os.path.join(HERE, "srs_kat.json")))
off_l, off_g2 = 4 + n * 64, 4 + 2 * n * 64
assert len(raw) == 33028 and raw[:4].hex() == kat["k_le"]
assert all(raw[4 + 64 * int(i): 4 + 64 * (int(i) + 1)].hex() == v for i, v in kat["g"].items())
assert all(raw[off_l + 64 * int(i): off_l + 64 * (int(i) + 1)].hex() == v for i, v in kat["g_lagrange"].items())
assert raw[off_g2: off_g2 + 128].hex() == kat["g2"] and raw[off_g2 + 128:].hex() == kat["s_g2"]
open(os.path.join(HERE, "kzg_bn254_8.srs"), "wb").write(raw)
print("ok", len(raw))

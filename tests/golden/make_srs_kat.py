"""Extracts a small known-answer set from the reference's only binary fixture,
halo2_verifier/params/kzg_bn254_8.srs (33,028 B, upstream PSE RawBytes layout:
u32le k | 2^k G1 g | 2^k G1 g_lagrange | G2 g2 | G2 s_g2, coordinates in Montgomery form),
of which tests/golden/kzg_bn254_8.srs is a copy (make_srs_fixture.py); the output
tests/golden/srs_kat.json is committed.  Only raw bytes are copied, no interpretation."""
import json, os, sys
SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "kzg_bn254_8.srs")
raw = open(SRC, "rb").read()
assert len(raw) == 33028
n = 256
off_l = 4 + n * 64
off_g2 = 4 + 2 * n * 64
kat = {
    "source": "halo2_verifier/params/kzg_bn254_8.srs",
    "k_le": raw[:4].hex(),
    "g": {str(i): raw[4 + 64 * i: 4 + 64 * (i + 1)].hex() for i in (0, 1, 2, 3, 255)},
    "g_lagrange": {str(i): raw[off_l + 64 * i: off_l + 64 * (i + 1)].hex() for i in (0, 1, 2, 255)},
    "g2": raw[off_g2: off_g2 + 128].hex(),
    "s_g2": raw[off_g2 + 128: off_g2 + 256].hex(),
}
json.dump(kat, open(os.path.join(os.path.dirname(__file__), "srs_kat.json"), "w"), indent=1)
print("ok")

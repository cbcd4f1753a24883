"""Derived parameters vs the tables the reference hard-codes, as recorded from its headers in
tests/golden/ref_params.json (tests/golden/make_golden.py params).  Roots of unity, Montgomery
constants and generators used by this repo are re-derived from first principles and merely
compared here."""
import json
import os
import re

GOLDEN = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_params.json")))


def _small_table(field, name):
    """ntt/parameters/{goldilocks,baby_bear}.h"""
    return [int(v, 16) for v in GOLDEN["ntt"][field][name]]


def test_goldilocks_roots(oracle):
    p = 2**64 - 2**32 + 1
    fwd = _small_table("goldilocks", "forward_roots_of_unity")
    inv = _small_table("goldilocks", "inverse_roots_of_unity")
    dsi = _small_table("goldilocks", "domain_size_inverse")
    for lg in range(33):
        assert oracle.lib().oracle_gl64_root(lg, 0) == fwd[lg]
        assert oracle.lib().oracle_gl64_root(lg, 1) == inv[lg]
        assert pow(2, -lg, p) == dsi[lg]
    assert fwd[32] == 0x185629dcda58878c == pow(7, (p - 1) >> 32, p)   # value hard-wired in ff/gl64.cuh


def test_babybear_roots(oracle):
    p, R = 0x78000001, 1 << 32
    fwd = _small_table("baby_bear", "forward_roots_of_unity")
    inv = _small_table("baby_bear", "inverse_roots_of_unity")
    dsi = _small_table("baby_bear", "domain_size_inverse")
    for lg in range(28):
        assert oracle.lib().oracle_bb31_root(lg, 0) * R % p == fwd[lg]     # tables are Montgomery words
        assert oracle.lib().oracle_bb31_root(lg, 1) * R % p == inv[lg]
        assert pow(2, -lg, p) * R % p == dsi[lg]
    assert fwd[27] * pow(R, -1, p) % p == 137


def test_msm_field_constants():
    """sppark_b200/csrc/ff/fields.cuh (generated) vs ff/bls12-381.hpp:14-52, ff/pasta.hpp:14-50."""
    gen = open(os.path.join(os.path.dirname(__file__), "..", "sppark_b200", "csrc", "ff", "fields.cuh")).read()

    def ours(struct, name):
        blk = gen.split(f"struct {struct}_params")[1].split("typedef")[0]
        m = re.search(r"%s\(int i\) \{ constexpr uint32_t t\[\d+\] = \{(.*?)\}" % name, blk)
        return [int(x.rstrip("u"), 16) for x in m.group(1).split(", ")]

    def theirs(header, name):
        """32-bit words of a device-side constant of ff/<header>.hpp"""
        return [int(v, 16) for v in GOLDEN["ff"][header][name]]

    b = "bls12-381"
    assert ours("bls12_381_fp", "P") == theirs(b, "BLS12_381_P")
    assert ours("bls12_381_fp", "RR") == theirs(b, "BLS12_381_RR")
    assert ours("bls12_381_fp", "ONE") == theirs(b, "BLS12_381_one")
    assert ours("bls12_381_fr", "P") == theirs(b, "BLS12_381_r")
    assert ours("bls12_381_fr", "ONE") == theirs(b, "BLS12_381_rone")
    q = "pasta"
    assert ours("pallas_fp", "P") == theirs(q, "Pallas_P")
    assert ours("pallas_fp", "RR") == theirs(q, "Pallas_RR")
    assert ours("pallas_fp", "ONE") == theirs(q, "Pallas_one")
    assert ours("vesta_fp", "P") == theirs(q, "Vesta_P")
    assert ours("vesta_fp", "ONE") == theirs(q, "Vesta_one")
    assert "M0 = 0xfffcfffdu" in gen.split("struct bls12_381_fp_params")[1].split("typedef")[0]
    # ff/alt_bn128.hpp:13-47, ff/bls12-377.hpp:13-51
    a = "alt_bn128"
    assert ours("bn254_fp", "P") == theirs(a, "ALT_BN128_P")
    assert ours("bn254_fp", "RR") == theirs(a, "ALT_BN128_RR")
    assert ours("bn254_fp", "ONE") == theirs(a, "ALT_BN128_one")
    assert ours("bn254_fr", "P") == theirs(a, "ALT_BN128_r")
    assert ours("bn254_fr", "RR") == theirs(a, "ALT_BN128_rRR")
    assert ours("bn254_fr", "ONE") == theirs(a, "ALT_BN128_rone")
    assert "M0 = 0xe4866389u" in gen.split("struct bn254_fp_params")[1].split("typedef")[0]
    assert "M0 = 0xefffffffu" in gen.split("struct bn254_fr_params")[1].split("typedef")[0]
    c = "bls12-377"
    assert ours("bls12_377_fp", "P") == theirs(c, "BLS12_377_P")
    assert ours("bls12_377_fp", "RR") == theirs(c, "BLS12_377_RR")
    assert ours("bls12_377_fp", "ONE") == theirs(c, "BLS12_377_one")
    assert ours("bls12_377_fr", "P") == theirs(c, "BLS12_377_r")
    assert ours("bls12_377_fr", "ONE") == theirs(c, "BLS12_377_rone")


def test_256bit_ntt_roots():
    """group_gen / 2^32-th roots of unity of the 256-bit NTT fields: derived (tools/gen_fields.py,
    oracle/ntt.c) vs ntt/parameters/{bls12_381,pallas,vesta}.h."""
    def table(name):
        out = {k: [int(v, 16) for v in vs] for k, vs in GOLDEN["ntt256"][name].items()}
        out["group_gen"] = out["group_gen"][0]
        return out
    R = 1 << 256
    for name, p, g, S in (("bls12_381", 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001, 7, 32),
                          ("vesta", 0x40000000000000000000000000000000224698fc0994a8dd8c46eb2100000001, 5, 32),
                          ("pallas", 0x40000000000000000000000000000000224698fc094cf91b992d30ed00000001, 5, 32),
                          ("alt_bn128", 0x30644e72e131a029b85045b68181585d2833e84879b9709143e1f593f0000001, 5, 28),
                          ("bls12_377", 0x12ab655e9a2ca55660b44d1e5c37b00159aa76fed00000010a11800000000001, 22, 47)):
        t = table(name)
        assert t["group_gen"] == g * R % p
        assert len(t["forward_roots_of_unity"]) == S + 1
        w = pow(g, (p - 1) >> S, p)
        for lg in range(S + 1):
            assert t["forward_roots_of_unity"][lg] == pow(w, 1 << (S - lg), p) * R % p
            assert t["domain_size_inverse"][lg] == pow(2, -lg, p) * R % p


def test_pasta_shim_constants():
    """oracle/shim/pasta_t.hpp (host field types for the reference's Pasta MSM build) vs the
    device-side tables of ff/pasta.hpp:12-50, and the Montgomery factors vs -p^-1 mod 2^64."""
    shim = open(os.path.join(os.path.dirname(__file__), "..", "oracle", "shim", "pasta_t.hpp")).read()

    def shim_words(name):
        m = re.search(r"static const vec256 %s = \{(.*?)\};" % name, shim, re.S)
        words = []
        for v in re.findall(r"TO_LIMB_T\((0x[0-9a-f]+)\)", m.group(1)):
            v = int(v, 16)
            words += [v & 0xFFFFFFFF, v >> 32]
        return words

    def ref_words(name):
        return [int(v, 16) for v in GOLDEN["ff"]["pasta"][name]]

    for ours, ref in (("Pallas_P", "Pallas_P"), ("Pallas_RR", "Pallas_RR"), ("Pallas_ONE", "Pallas_one"),
                      ("Vesta_P", "Vesta_P"), ("Vesta_RR", "Vesta_RR"), ("Vesta_ONE", "Vesta_one")):
        assert shim_words(ours) == ref_words(ref), ours
    for name, m0 in (("Pallas_P", 0x992d30ecffffffff), ("Vesta_P", 0x8c46eb20ffffffff)):
        w = shim_words(name)
        p = sum(v << (32 * i) for i, v in enumerate(w))
        assert (-pow(p, -1, 2**64)) % 2**64 == m0
        assert "0x%016xu" % m0 in shim
        assert m0 & 0xFFFFFFFF == 0xFFFFFFFF        # ff/pasta.hpp:51: Pasta_M0 = 0xffffffff

"""Pins the CPU oracle (runs without a GPU):
  - field arithmetic vs Python big integers and vs the constants the reference hard-codes
  - C restatement of Pippenger == naive double-and-add == the reference's own CPU
    msm/pippenger.hpp (golden vectors generated from oracle/_ref, tests/golden/make_golden.py)
  - NTT: fast == O(n^2) definition, and == the reference's own CUDA NTT / MSM outputs recorded
    on a B200 (tests/golden/*_ref_gpu.npz)."""
import os
import random

import numpy as np
import pytest

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
R_BLS = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001


def test_field_arithmetic_vs_python(oracle):
    rnd = random.Random(1)
    for name in ("bls12_381_fp", "bls12_381_fr", "pallas_fp", "vesta_fp", "bn254_fp", "bn254_fr",
                 "bls12_377_fp", "bls12_377_fr"):
        c = oracle.ff_consts(name)
        p, n = c["p"], c["n"]
        R = 1 << (64 * n)
        assert c["one"] == R % p and c["rr"] == R * R % p
        assert (c["m0"] * p + 1) % (1 << 64) == 0
        for _ in range(200):
            a, b = rnd.randrange(p), rnd.randrange(p)
            assert oracle.ff_op(name, "mul", a, b) == a * b * pow(R, -1, p) % p
            assert oracle.ff_op(name, "add", a, b) == (a + b) % p
            assert oracle.ff_op(name, "sub", a, b) == (a - b) % p
            assert oracle.ff_op(name, "to_mont", a) == a * R % p
            assert oracle.ff_op(name, "from_mont", a) == a * pow(R, -1, p) % p
        a = rnd.randrange(1, p)
        assert oracle.ff_op(name, "inv", a * R % p) == pow(a, -1, p) * R % p


def test_reference_constants(oracle):
    """ff/bls12-381.hpp:100-139 hard-codes these; the oracle derives them."""
    c = oracle.ff_consts("bls12_381_fp")
    assert c["m0"] == 0x89f3fffcfffcfffd
    assert c["rr"] & 0xFFFFFFFFFFFFFFFF == 0xf4df1f341c341746
    assert c["one"] & 0xFFFFFFFFFFFFFFFF == 0x760900000002fffd
    c = oracle.ff_consts("bls12_381_fr")
    assert c["m0"] == 0xfffffffeffffffff
    assert c["one"] >> 192 == 0x1824b159acc5056f


@pytest.mark.parametrize("curve", ["bls12_381", "pallas", "vesta", "bn254", "bls12_377"])
def test_generated_points_on_curve(oracle, curve):
    pts = oracle.gen_points(curve, 40)
    assert all(oracle.on_curve(curve, p) for p in pts)
    assert len({tuple(p) for p in pts}) == 40


R_OF = {"bn254": 0x30644e72e131a029b85045b68181585d2833e84879b9709143e1f593f0000001,
        "bls12_377": 0x12ab655e9a2ca55660b44d1e5c37b00159aa76fed00000010a11800000000001}


@pytest.mark.parametrize("curve", ["bn254", "bls12_377"])
def test_bn254_bls12_377_oracle(oracle, curve):
    """group order, naive == Pippenger (serial and threaded), and the golden recorded from the
    reference's own CUDA MSM for these curves on a B200 (tests/golden/make_golden.py curves2)."""
    r = R_OF[curve]
    nl = oracle.CURVE_LIMBS[oracle.CURVES[curve]]
    base = oracle.gen_points(curve, 32)
    inf = oracle.msm(curve, base[3:4], np.array([oracle.int_to_limbs(r, 4)], dtype=np.uint64), "naive")
    assert not inf[2 * nl:].any()
    n = 300
    pts = base[np.arange(n) % 32].copy()
    pts[3] = 0
    sc = _sc(n, 5, r)
    a = oracle.jac_to_affine(curve, oracle.msm(curve, pts, sc, "naive"))
    b = oracle.jac_to_affine(curve, oracle.msm(curve, pts, sc, "serial"))
    c = oracle.jac_to_affine(curve, oracle.msm(curve, pts, sc, "pippenger", ncpus=4))
    assert np.array_equal(a, b) and np.array_equal(a, c) and oracle.on_curve(curve, a)
    path = os.path.join(GOLD, "msm_curves2_ref_gpu.npz")
    if not os.path.exists(path):
        pytest.skip("golden not recorded")
    g = np.load(path)
    for k in range(int(g[f"{curve}_ncases"])):
        p = g[f"{curve}_points{k}"].copy()
        p[p[:, 2 * nl] != 0, :2 * nl] = 0                    # flagged rows are infinity
        got = oracle.jac_to_affine(curve, oracle.msm(curve, np.ascontiguousarray(p[:, :2 * nl]), g[f"{curve}_scalars{k}"]))
        assert np.array_equal(got, oracle.jac_to_affine(curve, g[f"{curve}_out{k}"])), k


@pytest.mark.parametrize("curve", ["pallas", "vesta"])
def test_pasta_oracle_matches_reference_gpu_golden(oracle, curve):
    """The oracle's Pallas / Vesta MSM against the reference's own CUDA MSM templates run for these
    curves on a B200 (ff/pasta.hpp:82-103 through oracle/ref_msm_g1.cu with the host field types of
    oracle/shim/pasta_t.hpp; tests/golden/make_golden.py pasta) -- this is what pins the Pasta
    oracle to the reference rather than to its own definition."""
    nl = oracle.CURVE_LIMBS[oracle.CURVES[curve]]
    g = np.load(os.path.join(GOLD, "msm_pasta_ref_gpu.npz"))
    assert int(g[f"{curve}_ncases"]) >= 5
    for k in range(int(g[f"{curve}_ncases"])):
        p = g[f"{curve}_points{k}"].copy()
        p[p[:, 2 * nl] != 0, :2 * nl] = 0                    # flagged rows are infinity
        got = oracle.jac_to_affine(curve, oracle.msm(curve, np.ascontiguousarray(p[:, :2 * nl]), g[f"{curve}_scalars{k}"]))
        want = oracle.jac_to_affine(curve, g[f"{curve}_out{k}"])
        assert np.array_equal(got, want) and oracle.on_curve(curve, want), k


def _sc(n, seed, r=R_BLS):
    rnd = random.Random(seed)
    return np.array([[(v >> (64 * i)) & (2**64 - 1) for i in range(4)]
                     for v in (rnd.randrange(r) for _ in range(n))], dtype=np.uint64).reshape(n, 4)


@pytest.mark.parametrize("n", [1, 2, 31, 32, 33, 193, 600])
def test_pippenger_serial_threaded_naive_agree(oracle, n):
    pts = oracle.gen_points("bls12_381", 32)[np.arange(n) % 32].copy()
    if n > 3:
        pts[3] = 0
    sc = _sc(n, n)
    aff = lambda j: tuple(oracle.jac_to_affine("bls12_381", j))  # noqa: E731
    a = aff(oracle.msm("bls12_381", pts, sc, "naive"))
    assert a == aff(oracle.msm("bls12_381", pts, sc, "serial"))
    assert a == aff(oracle.msm("bls12_381", pts, sc, "pippenger", ncpus=5))
    assert oracle.on_curve("bls12_381", np.array(a, dtype=np.uint64))


def test_oracle_matches_reference_cpu_golden(oracle):
    g = np.load(os.path.join(GOLD, "msm_ref_cpu.npz"))
    for n in (1, 2, 33, 200, 1000):
        got = oracle.jac_to_affine("bls12_381", oracle.msm("bls12_381", g[f"pts_{n}"], g[f"sc_{n}"], "pippenger", ncpus=4))
        assert np.array_equal(got, g[f"affine_{n}"]), n


def test_oracle_matches_reference_cpu_live(oracle):
    """The reference's CPU msm/pippenger.hpp on 700 points (recorded in msm_ref_cpu_n700.npz by
    tests/golden/make_golden.py cpu) vs the oracle's serial path."""
    n = 700
    pts = oracle.gen_points("bls12_381", 50)[np.arange(n) % 50].copy()
    sc = _sc(n, 3)
    g = np.load(os.path.join(GOLD, "msm_ref_cpu_n700.npz"))
    assert np.array_equal(g["pts"], pts) and np.array_equal(g["sc"], sc)
    assert np.array_equal(g["affine"], oracle.jac_to_affine("bls12_381", oracle.msm("bls12_381", pts, sc, "serial")))


def test_oracle_matches_reference_gpu_golden_msm(oracle):
    path = os.path.join(GOLD, "msm_ref_gpu.npz")
    if not os.path.exists(path):
        pytest.skip("reference-GPU golden not recorded yet")
    g = np.load(path)
    for n in (1, 2, 33, 200, 1000):
        got = oracle.jac_to_affine("bls12_381", oracle.msm("bls12_381", g[f"pts_{n}"], g[f"sc_{n}"], "pippenger", ncpus=4))
        assert np.array_equal(got, g[f"affine_{n}"]), n


@pytest.mark.parametrize("field", ["gl64", "bb31"])
def test_ntt_fast_equals_definition(oracle, field):
    rng = np.random.default_rng(5)
    fn = oracle.ntt_gl64 if field == "gl64" else oracle.ntt_bb31
    p, dt = (2**64 - 2**32 + 1, np.uint64) if field == "gl64" else (0x78000001, np.uint32)
    for lg in range(1, 10):
        x = rng.integers(0, p, size=1 << lg, dtype=dt)
        for order in range(5):
            for inv in (False, True):
                for coset in (False, True):
                    assert np.array_equal(fn(x, order, inv, coset, "dft"), fn(x, order, inv, coset, "fast"))
        assert np.array_equal(fn(fn(x, oracle.NR), oracle.RN, True), x)
        assert np.array_equal(fn(fn(x, oracle.NN, False, True), oracle.NN, True, True), x)


def test_ntt_small_known_answers(oracle):
    # NTT of a delta is all ones; of all-ones is n*delta; lg=1 is (a+b, a-b)
    p = 2**64 - 2**32 + 1
    x = np.zeros(16, dtype=np.uint64); x[0] = 1
    assert (oracle.ntt_gl64(x) == 1).all()
    y = oracle.ntt_gl64(np.ones(16, dtype=np.uint64))
    assert y[0] == 16 and not y[1:].any()
    z = oracle.ntt_gl64(np.array([5, 7], dtype=np.uint64))
    assert list(z) == [12, p - 2]
    # X[1] of (0,1,0,0) is the 4th root of unity 2^48 (ntt/parameters/goldilocks.h:93)
    w = oracle.ntt_gl64(np.array([0, 1, 0, 0], dtype=np.uint64))
    assert int(w[1]) == 1 << 48


def test_oracle_matches_reference_gpu_golden_ntt(oracle):
    """Goldilocks (lg 1..10) and BabyBear (lg 1..12): every order x direction x type of the
    reference's own CUDA NTT, recorded on a B200 with ONE reference library per process
    (tests/golden/make_golden.py explains why that matters), bit for bit."""
    path = os.path.join(GOLD, "ntt_ref_gpu.npz")
    if not os.path.exists(path):
        pytest.skip("reference-GPU golden not recorded yet")
    g = np.load(path)
    for field, fn, top in (("gl64", oracle.ntt_gl64, 10), ("bb31", oracle.ntt_bb31, 12)):
        for lg in range(1, top + 1):
            x = g[f"{field}_in_{lg}"]
            # the reference's own protocol holds in the recording: NN == RR
            assert np.array_equal(g[f"{field}_out_{lg}_000"], g[f"{field}_out_{lg}_300"])
            for order in range(4):
                for d in range(2):
                    for t in range(2):
                        assert np.array_equal(fn(x, order, bool(d), bool(t)), g[f"{field}_out_{lg}_{order}{d}{t}"]), \
                            (field, lg, order, d, t)


def test_oracle_matches_reference_gpu_golden_ntt256(oracle):
    """BLS12-381 scalar-field NTT (the reference's 256-bit "wide" kernels) recorded on a B200,
    lg 1..10, every order x direction x type."""
    path = os.path.join(GOLD, "ntt256_ref_gpu.npz")
    if not os.path.exists(path):
        pytest.skip("reference-GPU golden not recorded yet")
    g = oracle.ntt256_golden(path)
    for lg in range(1, 11):
        x = g[f"in_{lg}"]
        for order in range(4):
            for d in range(2):
                for t in range(2):
                    if lg > 8 and t == 1 and order in (1, 2):
                        continue                                          # keep the CPU suite short
                    assert np.array_equal(oracle.ntt_ff("bls12_381_fr", x, order, bool(d), bool(t)),
                                          g[f"out_{lg}_{order}{d}{t}"]), (lg, order, d, t)


@pytest.mark.parametrize("field", ["bls12_381_fr", "pallas_fp", "vesta_fp"])
def test_ntt256_fast_equals_definition(oracle, field):
    rnd = random.Random(3)
    p = oracle.ff_consts(field)["p"]
    for lg in range(1, 7):
        x = np.array([oracle.int_to_limbs(rnd.randrange(p), 4) for _ in range(1 << lg)], dtype=np.uint64)
        for order in range(5):
            for inv in (False, True):
                for coset in (False, True):
                    assert np.array_equal(oracle.ntt_ff(field, x, order, inv, coset, "dft"),
                                          oracle.ntt_ff(field, x, order, inv, coset, "fast"))
        assert np.array_equal(oracle.ntt_ff(field, oracle.ntt_ff(field, x, oracle.NR), oracle.RN, True), x)


def test_oracle_lde_matches_reference_gpu_golden(oracle):
    """NTT::LDE of the reference (Goldilocks) recorded on a B200 vs the oracle's definition."""
    path = os.path.join(GOLD, "lde_ref_gpu.npz")
    if not os.path.exists(path):
        pytest.skip("reference-GPU golden not recorded yet")
    g = np.load(path)
    for lg, lb in ((1, 1), (3, 1), (6, 2), (10, 1), (12, 3)):
        ext, _ = oracle.lde("gl64", g[f"in_{lg}_{lb}"], lb)
        assert np.array_equal(ext, g[f"out_{lg}_{lb}"]), (lg, lb)

"""GPU parity for the MSM path: CUDA through the C-ABI vs the CPU oracle.  MSM results are
compared as group elements (affine-normalised), as the reference's own tests do
(poc/msm-cuda/tests/msm.rs:27-38); field arithmetic is compared bit-exactly."""
import random

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

R_BLS = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001
FIELDS = [("bls12_381_fp", 0, 6), ("bls12_381_fr", 1, 4), ("pallas_fp", 2, 4), ("vesta_fp", 3, 4),
          ("bn254_fp", 4, 4), ("bn254_fr", 5, 4), ("bls12_377_fp", 6, 6), ("bls12_377_fr", 7, 4)]


def _limbs(x, n):
    return [(x >> (64 * i)) & 0xFFFFFFFFFFFFFFFF for i in range(n)]


def _int(row):
    return sum(int(v) << (64 * i) for i, v in enumerate(row))


@pytest.mark.parametrize("name,fid,nl", FIELDS)
def test_field_kat_ptx(oracle, name, fid, nl):
    """PTX Montgomery arithmetic vs Python big integers (bit-exact), incl. edge values."""
    from sppark_b200 import msm
    p = oracle.ff_consts(name)["p"]
    R = 1 << (64 * nl)
    rnd = random.Random(fid)
    vals = [0, 1, p - 1, p - 2, 2, (1 << (64 * nl - 1)) % p, R % p] + [rnd.randrange(p) for _ in range(2000)]
    a = np.array([_limbs(v, nl) for v in vals], dtype=np.uint64)
    b = np.array([_limbs(v, nl) for v in reversed(vals)], dtype=np.uint64)
    Rinv = pow(R, -1, p)
    for op, fn in (("mul", lambda x, y: x * y * Rinv % p), ("add", lambda x, y: (x + y) % p),
                   ("sub", lambda x, y: (x - y) % p), ("sqr", lambda x, y: x * x * Rinv % p),
                   ("mul_shared", lambda x, y: x * y * Rinv % p), ("sqr_shared", lambda x, y: x * x * Rinv % p),
                   ("msub_shared", lambda x, y: (x * y - y * (x * x * Rinv % p)) * Rinv % p)):
        r = msm.selftest_field(fid, op, a, b)
        for i in range(len(vals)):
            assert _int(r[i]) == fn(vals[i], vals[len(vals) - 1 - i]), (name, op, i)


def _scalars(n, seed, r=R_BLS):
    rnd = random.Random(seed)
    return np.array([_limbs(rnd.randrange(r), 4) for _ in range(n)], dtype=np.uint64).reshape(n, 4)


def _same_point(oracle, curve, a, b):
    return np.array_equal(oracle.jac_to_affine(curve, a), oracle.jac_to_affine(curve, b))


@pytest.mark.parametrize("n", [1, 2, 31, 32, 33, 193, 1000, 4096, 1 << 14])
def test_bls12_381_msm_matches_oracle(oracle, n):
    from sppark_b200 import msm
    base = oracle.gen_points("bls12_381", min(n, 2048))
    pts = base[np.arange(n) % base.shape[0]].copy()
    if n > 3:
        pts[3] = 0                                  # point at infinity, as util.rs:29-31 plants one
    sc = _scalars(n, n)
    got = msm.multi_scalar_mult(pts, sc)
    want = oracle.msm("bls12_381", pts, sc, "pippenger", ncpus=8)
    assert _same_point(oracle, "bls12_381", got, want)


@pytest.mark.parametrize("kind", ["zero", "one", "r_minus_1", "all_same", "pm_pairs", "one_heavy"])
def test_bls12_381_msm_adversarial(oracle, kind):
    from sppark_b200 import msm
    n = 5000
    base = oracle.gen_points("bls12_381", 16)
    pts = base[np.arange(n) % 16].copy()
    p = oracle.ff_consts("bls12_381_fp")["p"]
    if kind == "zero":
        sc = np.zeros((n, 4), dtype=np.uint64)
    elif kind == "one":
        sc = np.tile(np.array(_limbs(1, 4), dtype=np.uint64), (n, 1))
    elif kind == "r_minus_1":
        sc = np.tile(np.array(_limbs(R_BLS - 1, 4), dtype=np.uint64), (n, 1))
    elif kind == "all_same":
        sc = np.tile(np.array(_limbs(0x1234567890ABCDEF1234567890ABCDEF1234567890ABCDEF, 4), dtype=np.uint64), (n, 1))
    elif kind == "pm_pairs":
        sc = np.tile(np.array(_limbs(12345, 4), dtype=np.uint64), (n, 1))
        for i in range(1, n, 2):                    # odd rows: the negated previous point
            pts[i, :6] = pts[i - 1, :6]
            pts[i, 6:] = np.array(_limbs(p - _int(pts[i - 1, 6:]), 6), dtype=np.uint64)
    else:
        sc = _scalars(n, 99)
        sc[: n // 2] = sc[0]                        # half of the points share every bucket
    got = msm.multi_scalar_mult(pts, sc)
    want = oracle.msm("bls12_381", pts, sc, "pippenger", ncpus=8)
    assert _same_point(oracle, "bls12_381", got, want)
    if kind in ("zero", "pm_pairs"):
        assert not got[12:].any()                   # infinity encodes as Z == 0


def test_mult_pippenger_inf_layout(oracle):
    """arkworks G1Affine layout: 104-byte rows, infinity flag in the byte after Y
    (pippenger_inf.cu:28-34, ec/affine_t.hpp:91-96)."""
    from sppark_b200 import msm
    n = 3000
    base = oracle.gen_points("bls12_381", 128)
    pts = np.zeros((n, 13), dtype=np.uint64)
    pts[:, :12] = base[np.arange(n) % 128]
    pts[::7, 12] = 1                                # flagged rows keep garbage coordinates on purpose
    sc = _scalars(n, 5)
    got = msm.multi_scalar_mult_arkworks(pts, sc)
    clean = pts[:, :12].copy()
    clean[::7] = 0
    want = oracle.msm("bls12_381", clean, sc, "pippenger", ncpus=8)
    assert _same_point(oracle, "bls12_381", got, want)


@pytest.mark.parametrize("curve,cid", [("pallas", 1), ("vesta", 2)])
def test_pasta_msm_matches_oracle(oracle, curve, cid):
    from sppark_b200 import msm
    n = 6000
    r = oracle.ff_consts("vesta_fp" if curve == "pallas" else "pallas_fp")["p"]
    base = oracle.gen_points(curve, 256)
    pts = base[np.arange(n) % 256].copy()
    sc = _scalars(n, 11, r)
    got = msm.msm(cid, pts, sc)
    want = oracle.msm(curve, pts, sc, "pippenger", ncpus=8)
    assert _same_point(oracle, curve, got, want)
    # ... and against the reference's own CUDA MSM templates instantiated for this curve, recorded
    # on a B200 (tests/golden/make_golden.py pasta: ff/pasta.hpp through oracle/ref_msm_g1.cu):
    # arkworks-style rows with infinity flags, scalars below the group order incl. 0 and r - 1
    import os
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "msm_pasta_ref_gpu.npz"))
    for k in range(int(g[f"{curve}_ncases"])):
        got = msm.msm(cid, np.ascontiguousarray(g[f"{curve}_points{k}"]), np.ascontiguousarray(g[f"{curve}_scalars{k}"]))
        assert _same_point(oracle, curve, got, g[f"{curve}_out{k}"]), k


@pytest.mark.parametrize("curve,cid,fr", [("bn254", 4, "bn254_fr"), ("bls12_377", 5, "bls12_377_fr")])
def test_bn254_bls12_377_msm(oracle, curve, cid, fr):
    """The msm crate's other two curve features (poc/msm-cuda/Cargo.toml: bn254, bls12_377): vs the
    oracle on packed and arkworks rows, scalars plain and in Montgomery form, device-resident
    entry + generated points, and vs the reference's own CUDA MSM recorded on a B200."""
    import os
    import torch
    from sppark_b200 import msm
    r = oracle.ff_consts(fr)["p"]
    nl = oracle.CURVE_LIMBS[oracle.CURVES[curve]]
    for n in (1, 33, 5000, 1 << 15):
        base = oracle.gen_points(curve, min(n, 512))
        pts = base[np.arange(n) % base.shape[0]].copy()
        if n > 3:
            pts[3] = 0
        sc = _scalars(n, n + cid, r)
        want = oracle.msm(curve, pts, sc, "pippenger", ncpus=8)
        assert _same_point(oracle, curve, msm.msm(cid, pts, sc), want), n
        ark = np.zeros((n, 2 * nl + 1), dtype=np.uint64)
        ark[:, :2 * nl] = pts
        if n > 7:
            ark[7, 2 * nl] = 1
            pts[7] = 0
            want = oracle.msm(curve, pts, sc, "pippenger", ncpus=8)
        assert _same_point(oracle, curve, msm.msm(cid, ark, sc), want), n
        if n == 5000:
            mont = np.array([_limbs(oracle.ff_op(fr, "to_mont", _int(row)), 4) for row in sc], dtype=np.uint64)
            assert _same_point(oracle, curve, msm.msm(cid, ark, mont, mont=True), want)
    gen = msm.generate_points_dev(cid, 300)
    assert np.array_equal(gen.cpu().numpy().view(np.uint64), oracle.gen_points(curve, 300))
    sc = _scalars(300, 3, r)
    got = msm.msm_dev(cid, gen, torch.from_numpy(sc.view(np.int64)).cuda())
    assert _same_point(oracle, curve, got, oracle.msm(curve, oracle.gen_points(curve, 300), sc, "pippenger", ncpus=8))
    path = os.path.join(os.path.dirname(__file__), "golden", "msm_curves2_ref_gpu.npz")
    if os.path.exists(path):
        g = np.load(path)
        for k in range(int(g[f"{curve}_ncases"])):
            got = msm.msm(cid, np.ascontiguousarray(g[f"{curve}_points{k}"]), np.ascontiguousarray(g[f"{curve}_scalars{k}"]))
            assert _same_point(oracle, curve, got, g[f"{curve}_out{k}"]), k


def test_bls12_381_msm_2pow20_folded(oracle):
    """2^20 points = 2^10 distinct points replicated: sum_i s_i P_(i mod m) equals the m-point MSM
    with scalars folded mod r, which the oracle finishes in seconds."""
    from sppark_b200 import msm
    n, m = 1 << 20, 1 << 10
    base = oracle.gen_points("bls12_381", m)
    pts = np.tile(base, (n // m, 1))
    rng = np.random.default_rng(42)
    sc = rng.integers(0, 2**64, size=(n, 4), dtype=np.uint64)
    sc[:, 3] >>= np.uint64(2)                         # < 2^254 < r
    got = msm.multi_scalar_mult(pts, sc)
    folded = np.zeros((m, 4), dtype=np.uint64)
    ints = [0] * m
    scl = sc.reshape(n // m, m, 4)
    for limb in range(4):
        col = scl[:, :, limb].astype(object).sum(axis=0)
        for j in range(m):
            ints[j] += int(col[j]) << (64 * limb)
    for j in range(m):
        folded[j] = _limbs(ints[j] % R_BLS, 4)
    want = oracle.msm("bls12_381", base, folded, "pippenger", ncpus=8)
    assert _same_point(oracle, "bls12_381", got, want)


def test_bls12_381_msm_2pow22_default_slicing(oracle):
    """2^22 points through mult_pippenger: the size from which the host pipeline cuts the input into
    N/16, N/8, N/4, 9N/16 slices copied while the previous slice is accumulated (msm_host.cuh);
    checked by folding the scalars of the replicated points onto the 2^10 distinct ones."""
    from sppark_b200 import msm
    n, m = 1 << 22, 1 << 10
    base = oracle.gen_points("bls12_381", m)
    pts = np.tile(base, (n // m, 1))
    pts[3] = 0
    rng = np.random.default_rng(22)
    sc = rng.integers(0, 2**64, size=(n, 4), dtype=np.uint64)
    sc[:, 3] >>= np.uint64(2)
    sc[3] = 0
    got = msm.multi_scalar_mult(pts, sc)
    halves = sc.reshape(n // m, m, 4).view(np.uint32).reshape(n // m, m, 8).astype(np.uint64).sum(axis=0)   # < 2^44 each
    folded = np.array([_limbs(sum(int(v) << (32 * k) for k, v in enumerate(row)) % R_BLS, 4) for row in halves], dtype=np.uint64)
    want = oracle.msm("bls12_381", base, folded, "pippenger", ncpus=8)
    assert _same_point(oracle, "bls12_381", got, want)


@pytest.mark.parametrize("curve,cid,fr", [("bls12_381", 0, "bls12_381_fr"), ("pallas", 1, "vesta_fp"), ("bn254", 4, "bn254_fr")])
def test_preloaded_points_context(oracle, curve, cid, fr):
    """sppark_b200_msm_ctx_*: points uploaded once (packed or arkworks rows), several scalar
    vectors against them, prefixes, Montgomery-form scalars; and the error paths."""
    from sppark_b200 import _lib, msm
    r = oracle.ff_consts(fr)["p"]
    nl = oracle.CURVE_LIMBS[oracle.CURVES[curve]]
    n = 1 << 15
    base = oracle.gen_points(curve, 256)
    pts = base[np.arange(n) % 256].copy()
    ark = np.zeros((n, 2 * nl + 1), dtype=np.uint64)
    ark[:, :2 * nl] = pts
    ark[11, 2 * nl] = 1
    ref = pts.copy()
    ref[11] = 0
    for layout, want_pts in ((pts, pts), (ark, ref)):
        ctx = msm.MsmContext(cid, layout)
        for seed, m in ((1, n), (2, n), (3, 1000), (4, 1)):
            sc = _scalars(m, seed, r)
            assert _same_point(oracle, curve, ctx.invoke(sc), oracle.msm(curve, want_pts[:m], sc, "pippenger", ncpus=8)), (seed, m)
        sc = _scalars(500, 9, r)
        mont = np.array([_limbs(oracle.ff_op(fr, "to_mont", _int(row)), 4) for row in sc], dtype=np.uint64)
        assert _same_point(oracle, curve, ctx.invoke(mont, mont=True), oracle.msm(curve, want_pts[:500], sc, "pippenger", ncpus=8))
        assert not ctx.invoke(np.zeros((0, 4), dtype=np.uint64)).any()          # no scalars: infinity
        with pytest.raises(_lib.SpparkError):
            ctx.invoke(_scalars(n + 1, 5, r))                                    # more scalars than points
        ctx.close()


def test_batched_affine_prereduction(oracle, monkeypatch):
    """SPPARK_B200_MSM_PAIR=1 (experimental, off by default; msm_pair.cuh): bucket lists halved by
    batched affine pair sums before the XYZZ accumulation.  Same group element as the oracle on
    random, replicated (tangent pairs), cancelling, heavy and sliced inputs."""
    from sppark_b200 import msm
    monkeypatch.setenv("SPPARK_B200_MSM_PAIR", "1")
    base = oracle.gen_points("bls12_381", 512)
    for n, seed in ((1, 1), (2, 2), (193, 3), (5000, 4), (1 << 16, 5)):
        pts = base[np.arange(n) % 512].copy()
        if n > 3:
            pts[3] = 0
        sc = _scalars(n, seed)
        assert _same_point(oracle, "bls12_381", msm.multi_scalar_mult(pts, sc), oracle.msm("bls12_381", pts, sc, "pippenger", ncpus=8)), n
    n = 3000
    sc = _scalars(n, 6)
    same = np.tile(base[7], (n, 1))                                   # one point, one scalar: tangents all the way
    s1 = np.tile(sc[0], (n, 1))
    assert _same_point(oracle, "bls12_381", msm.multi_scalar_mult(same, s1), oracle.msm("bls12_381", same, s1, "pippenger", ncpus=8))
    p = oracle.ff_consts("bls12_381_fp")["p"]
    pm = same.copy()
    pm[1::2, 6:] = _limbs(p - _int(same[0][6:]), 6)                  # (P, -P) pairs: everything cancels
    got = msm.multi_scalar_mult(pm, s1)
    assert not got[12:].any()
    mix = base[np.arange(n) % 16].copy()                              # few distinct points, few distinct scalars
    s2 = sc[np.arange(n) % 5].copy()
    assert _same_point(oracle, "bls12_381", msm.multi_scalar_mult(mix, s2), oracle.msm("bls12_381", mix, s2, "pippenger", ncpus=8))
    monkeypatch.setenv("SPPARK_B200_MSM_SLICES", "3")
    pts = base[np.arange(20000) % 512].copy()
    sc = _scalars(20000, 8)
    assert _same_point(oracle, "bls12_381", msm.multi_scalar_mult(pts, sc), oracle.msm("bls12_381", pts, sc, "pippenger", ncpus=8))
    monkeypatch.delenv("SPPARK_B200_MSM_SLICES")
    pal = oracle.gen_points("pallas", 64)[np.arange(4096) % 64].copy()
    scp = _scalars(4096, 9, oracle.ff_consts("vesta_fp")["p"])
    assert _same_point(oracle, "pallas", msm.msm(1, pal, scp), oracle.msm("pallas", pal, scp, "pippenger", ncpus=8))


def test_matches_reference_golden(oracle):
    """Same group element as the reference's CUDA mult_pippenger (recorded on a B200) and as its
    CPU msm/pippenger.hpp, on the committed inputs."""
    import os
    from sppark_b200 import msm
    for name in ("msm_ref_gpu.npz", "msm_ref_cpu.npz"):
        g = np.load(os.path.join(os.path.dirname(__file__), "golden", name))
        for n in (1, 2, 33, 200, 1000):
            got = msm.multi_scalar_mult(np.ascontiguousarray(g[f"pts_{n}"]), np.ascontiguousarray(g[f"sc_{n}"]))
            assert np.array_equal(oracle.jac_to_affine("bls12_381", got), g[f"affine_{n}"]), (name, n)


def test_generated_points_and_combine(oracle):
    from sppark_b200 import msm
    for curve, cid in (("bls12_381", 0), ("pallas", 1), ("vesta", 2)):
        pts = msm.generate_points_dev(cid, 300).cpu().numpy().view(np.uint64)
        assert np.array_equal(pts, oracle.gen_points(curve, 300))
    # combine: sum of Jacobian partials == MSM with unit scalars
    pts = oracle.gen_points("bls12_381", 5)
    one = np.tile(np.array(_limbs(1, 4), dtype=np.uint64), (5, 1))
    parts = np.stack([msm.multi_scalar_mult(pts[i:i + 1].copy(), one[i:i + 1].copy()) for i in range(5)])
    total = msm.combine(0, parts)
    want = oracle.msm("bls12_381", pts, one, "naive")
    assert _same_point(oracle, "bls12_381", total, want)


def test_device_resident_entry(oracle):
    import torch
    from sppark_b200 import msm
    n = 20000
    pts = oracle.gen_points("bls12_381", 500)[np.arange(n) % 500].copy()
    sc = _scalars(n, 77)
    got = msm.msm_dev(0, torch.from_numpy(pts.view(np.int64)).cuda(), torch.from_numpy(sc.view(np.int64)).cuda())
    want = oracle.msm("bls12_381", pts, sc, "pippenger", ncpus=8)
    assert _same_point(oracle, "bls12_381", got, want)


@pytest.mark.parametrize("nslices", [2, 3, 7])
def test_host_pipeline_slices(oracle, monkeypatch, nslices):
    """host-pointer path with the input cut into slices that share one bucket file"""
    from sppark_b200 import msm
    monkeypatch.setenv("SPPARK_B200_MSM_SLICES", str(nslices))
    n = 30011
    pts = np.zeros((n, 13), dtype=np.uint64)
    pts[:, :12] = oracle.gen_points("bls12_381", 97)[np.arange(n) % 97]
    pts[::11, 12] = 1
    sc = _scalars(n, nslices)
    sc[100:9000] = sc[7]                                # a heavy bucket in every window and slice
    clean = pts[:, :12].copy()
    clean[::11] = 0
    want = oracle.msm("bls12_381", clean, sc, "pippenger", ncpus=8)
    assert _same_point(oracle, "bls12_381", msm.multi_scalar_mult_arkworks(pts, sc), want)
    assert _same_point(oracle, "bls12_381", msm.multi_scalar_mult(clean, sc), want)


def test_pallas_msm_2pow21_folded(oracle):
    """BASELINE config 4 shape (Pallas, 2^21 points per GPU): folded check against the oracle."""
    from sppark_b200 import msm
    n, m = 1 << 21, 1 << 9
    r = oracle.ff_consts("vesta_fp")["p"]
    base = oracle.gen_points("pallas", m)
    pts = np.tile(base, (n // m, 1))
    rng = np.random.default_rng(4)
    sc = rng.integers(0, 2**64, size=(n, 4), dtype=np.uint64)
    sc[:, 3] >>= np.uint64(3)                         # < 2^253 < r
    got = msm.msm(1, pts, sc)
    ints = [0] * m
    scl = sc.reshape(n // m, m, 4)
    for limb in range(4):
        col = scl[:, :, limb].astype(object).sum(axis=0)
        for j in range(m):
            ints[j] += int(col[j]) << (64 * limb)
    folded = np.array([_limbs(v % r, 4) for v in ints], dtype=np.uint64)
    want = oracle.msm("pallas", base, folded, "pippenger", ncpus=8)
    assert _same_point(oracle, "pallas", got, want)


@pytest.mark.parametrize("kind", ["uniform_2pow16", "all_same_2pow20", "two_values_2pow20"])
def test_no_serialised_buckets(oracle, kind):
    """Guards the load balancing: neither the narrow top window of a small MSM nor a scalar
    distribution that puts every point into one bucket per window may end up on a single lane
    (a serial chain of 2^20 mixed adds takes ~10 s; the budget below is two orders above normal)."""
    import time
    import torch
    from sppark_b200 import msm
    n = 1 << (16 if kind == "uniform_2pow16" else 20)
    m = 1 << 10
    base = msm.generate_points_dev(0, m)
    dp = base.repeat(n // m, 1).contiguous()
    rng = np.random.default_rng(1)
    if kind == "uniform_2pow16":
        sc = rng.integers(0, 2**64, size=(n, 4), dtype=np.uint64)
        sc[:, 3] >>= np.uint64(2)
    elif kind == "all_same_2pow20":
        sc = np.tile(np.array(_limbs(0x0123456789ABCDEF0FEDCBA9876543210123456789ABCDEF0FEDCBA987654321 % R_BLS, 4),
                              dtype=np.uint64), (n, 1))
    else:
        sc = np.tile(np.array([_limbs(R_BLS - 5, 4), _limbs(3, 4)], dtype=np.uint64), (n // 2, 1))
    ds = torch.from_numpy(sc.view(np.int64)).cuda()
    msm.msm_dev(0, dp, ds)
    torch.cuda.synchronize()
    t = time.perf_counter()
    got = msm.msm_dev(0, dp, ds)
    dt = time.perf_counter() - t
    assert dt < 0.5, f"{kind}: {dt * 1e3:.0f} ms"
    # value check by folding onto the m distinct points
    ints = [0] * m
    scl = sc.reshape(n // m, m, 4)
    for limb in range(4):
        col = scl[:, :, limb].astype(object).sum(axis=0)
        for j in range(m):
            ints[j] += int(col[j]) << (64 * limb)
    folded = np.array([_limbs(v % R_BLS, 4) for v in ints], dtype=np.uint64)
    want = oracle.msm("bls12_381", base.cpu().numpy().view(np.uint64), folded, "pippenger", ncpus=8)
    assert _same_point(oracle, "bls12_381", got, want)


@pytest.mark.parametrize("curve,cid", [("bls12_381", 0), ("pallas", 1)])
def test_msm_sharded_c_abi(oracle, curve, cid):
    """sppark_b200_msm_sharded (single process, C ABI): chunks on device 0 one after the other, and
    on every visible device when there are several; same group element as the one-device call."""
    import torch
    from sppark_b200 import msm, parallel
    n = 50000
    r = R_BLS if curve == "bls12_381" else oracle.ff_consts("vesta_fp")["p"]
    base = oracle.gen_points(curve, 512)
    pts = base[np.arange(n) % 512].copy()
    pts[7] = 0
    sc = _scalars(n, 77, r)
    want = msm.msm(cid, pts, sc)
    for ids in ([0], [0, 0, 0], list(range(torch.cuda.device_count()))):
        got = parallel.msm_sharded_c(cid, pts, sc, ids)
        assert _same_point(oracle, curve, got, want), ids
    # ragged: fewer points than chunks
    got = parallel.msm_sharded_c(cid, pts[:2], sc[:2], [0, 0, 0, 0])
    assert _same_point(oracle, curve, got, msm.msm(cid, pts[:2], sc[:2]))


def test_scalar_bit_255_is_ignored_and_odd_strides_are_rejected(oracle):
    """Bits from nbits = 255 up are ignored, as in the reference's digit extraction
    (msm/pippenger.cuh:33-70): a scalar with bit 255 set gives the result of the scalar without it,
    whatever window width npoints selects.  Row strides that are not a multiple of 4 bytes are an
    argument error, not a device fault."""
    from sppark_b200 import _lib, msm
    for n in (100, 1 << 20):                          # c = 16 divides 256 around 2^20 points
        base = oracle.gen_points("bls12_381", 64)
        pts = base[np.arange(n) % 64].copy()
        sc = _scalars(n, 5 + n)
        hi = sc.copy()
        hi[::3, 3] |= np.uint64(1 << 63)
        assert _same_point(oracle, "bls12_381", msm.multi_scalar_mult(pts, hi), msm.multi_scalar_mult(pts, sc)), n
    raw = np.zeros(97 * 8 + 8, dtype=np.uint8)
    out = np.zeros(18, dtype=np.uint64)
    sc = _scalars(8, 1)
    err = _lib.lib().mult_pippenger_inf(out.ctypes.data, raw.ctypes.data, 8, sc.ctypes.data, 97)
    assert err.code != 0
    if err.message:
        _lib.lib().drop_error_message(err.message)


def test_bls12_381_msm_2pow26_equals_reference_gpu():
    """BASELINE config 3 at full size: the same group element as the reference's own CUDA
    mult_pippenger (its sources built for sm_100a, run on a B200 and recorded in
    msm_ref_gpu_2pow26.npz by tests/golden/make_golden.py msm_2pow26) on 2^26 points,
    compared with the library's own field arithmetic (cross-multiplied coordinates)."""
    import os
    import sys
    import torch
    from sppark_b200 import msm
    sys.path.insert(0, os.path.join(os.path.dirname(__file__), ".."))
    import bench
    theirs = np.load(os.path.join(os.path.dirname(__file__), "golden", "msm_ref_gpu_2pow26.npz"))["out"]
    n, m = 1 << 26, 1 << 16
    base = msm.generate_points_dev(msm.BLS12_381_G1, m).cpu().numpy().view(np.uint64)
    pts = np.empty((n, 12), dtype=np.uint64)
    pts.reshape(n // m, m, 12)[:] = base
    rng = np.random.default_rng(26)
    sc = np.empty((n, 4), dtype=np.uint64)
    for s in range(0, n, 1 << 22):
        sc[s:s + (1 << 22)] = rng.integers(0, 2**64, size=(1 << 22, 4), dtype=np.uint64)
    sc[:, 3] >>= np.uint64(2)
    ours = msm.multi_scalar_mult(pts, sc)
    assert bench._jac_equal(ours, theirs, msm)
    # and the size-independent property: folding the scalars onto the 2^16 distinct points
    folded = bench.fold_scalars(sc, m)
    small = msm.multi_scalar_mult(np.ascontiguousarray(base), folded)
    assert bench._jac_equal(ours, small, msm)
    del pts, sc
    torch.cuda.empty_cache()


def test_two_rank_nccl_bench_legs():
    """One process per GPU over NCCL (the launch the driver uses), when this box has two GPUs:
    sharded BLS12-381 and Pallas MSMs and the slab-sharded NTTs at reduced sizes; every leg's
    self-check must say ok."""
    import json
    import os
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU")
    root = os.path.join(os.path.dirname(__file__), "..")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", "29533", os.path.join(root, "bench.py"),
           "--gpus", "2", "--steps", "1", "--warmup", "3", "--lg-msm", "20", "--lg-ntt", "20", "--lg-pallas", "18", "--skip-cpu"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["n_gpus"] == 2 and line["check"].endswith("ok"), line["check"]
    assert line["pallas_msm"]["check"].endswith("ok"), line["pallas_msm"]
    assert line["e2e"]["same_result"] is True
    assert line["ntt"]["value"] > 0 and line["ntt"]["babybear_2pow27"]["value"] > 0

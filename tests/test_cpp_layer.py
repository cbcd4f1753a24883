"""The C++ surface (include/sppark_b200.hpp + include/compat/): layouts, that the reference's own
poc glue compiles UNMODIFIED against it, and -- on a GPU -- that what those builds compute equals
the oracle.  SURVEY.md section 8b, "C++-level names to keep"."""
import ctypes as C
import importlib.util
import os
import random
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CPP = os.path.join(ROOT, "tests", "cpp")
OUT = os.path.join(CPP, "_build")
R_BLS = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001
GL_P = 2**64 - 2**32 + 1


def _builder():
    spec = importlib.util.spec_from_file_location("build_cpp", os.path.join(CPP, "build_cpp.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


@pytest.mark.parametrize("feature", ["BLS12_381", "PALLAS", "VESTA", "BN254", "BLS12_377", "GOLDILOCKS", "BABY_BEAR"])
def test_layouts_compile(feature):
    subprocess.check_call(["g++", "-std=c++17", "-fsyntax-only", f"-DFEATURE_{feature}", "-I" + os.path.join(ROOT, "include"),
                           os.path.join(CPP, "layout_check.cpp")])


@pytest.mark.parametrize("feature", ["GOLDILOCKS", "BABY_BEAR", "BLS12_381"])
def test_polynomial_headers_forward(feature):
    """<polynomial/prefix_op.cuh>, <polynomial/div_by_x_minus_z.cuh>, <polynomial/evaluate.cuh> and
    <ff/batch_inversion.hpp> resolve under include/compat to the same-named templates over the C ABI"""
    src = open(os.path.join(CPP, "poly_compat_check.cpp")).read()
    if feature != "GOLDILOCKS":
        src = src.replace("<ff/goldilocks.hpp>", "<ff/baby_bear.hpp>" if feature == "BABY_BEAR" else "<ff/bls12-381.hpp>")
    subprocess.run(["g++", "-std=c++17", "-fsyntax-only", "-x", "c++", f"-DFEATURE_{feature}",
                    "-I" + os.path.join(ROOT, "include", "compat"), "-"], input=src, text=True, check=True)


def test_unbuilt_curves_are_refused_at_compile_time():
    r = subprocess.run(["g++", "-std=c++17", "-fsyntax-only", "-DFEATURE_MERSENNE31", "-I" + os.path.join(ROOT, "include"),
                        os.path.join(CPP, "layout_check.cpp")], capture_output=True, text=True)
    assert r.returncode != 0 and "not instantiated" in r.stderr


def test_example_links_against_the_library(lib):
    exe, exe_ntt = _builder().build_example()
    assert os.path.exists(exe) and os.path.exists(exe_ntt)


def test_reference_poc_glue_compiles_unmodified(lib):
    """poc/msm-cuda/cuda/pippenger.cu, pippenger_inf.cu and poc/ntt-cuda/cuda/ntt_api.cu, from where
    they lie, with plain g++ and -I include/compat: the reference's C++ callers switch libraries by
    switching the include path."""
    if not os.path.isdir("/root/reference"):
        pytest.skip("needs a checkout of the original project: its poc glue sources cannot be part of this repository")
    built = _builder().build_reference_glue()
    assert len(built) == 7
    syms = subprocess.check_output(["nm", "-D", os.path.join(OUT, "libdropin_msm.so")], text=True)
    assert " T mult_pippenger_inf" in syms and " T mult_pippenger_fp2_inf" in syms
    syms = subprocess.check_output(["nm", "-D", os.path.join(OUT, "libdropin_ntt_gl64.so")], text=True)
    assert " T compute_ntt" in syms


class RE(C.Structure):
    _fields_ = [("code", C.c_int), ("message", C.c_void_p)]


def _limbs(x, n=4):
    return [(x >> (64 * i)) & 0xFFFFFFFFFFFFFFFF for i in range(n)]


def _scalars(n, seed):
    rnd = random.Random(seed)
    return np.array([_limbs(rnd.randrange(R_BLS)) for _ in range(n)], dtype=np.uint64).reshape(n, 4)


@pytest.mark.gpu
@pytest.mark.parametrize("mont", [0, 1])
def test_cpp_example_msm(oracle, tmp_path, mont):
    """mult_pippenger<bucket_t>(out, points, n, scalars, mont, sizeof(affine_t)) from C++; mont = 1
    is the template's default in the reference: scalars arrive as Montgomery residues."""
    exe, _ = _builder().build_example()
    n = 3000
    base = oracle.gen_points("bls12_381", 128)
    pts = np.zeros((n, 13), dtype=np.uint64)
    pts[:, :12] = base[np.arange(n) % 128]
    pts[5, 12] = 1
    sc = _scalars(n, 31 + mont)
    send = sc
    if mont:
        send = np.array([_limbs(oracle.ff_op("bls12_381_fr", "to_mont", sum(int(v) << (64 * j) for j, v in enumerate(row))))
                         for row in sc], dtype=np.uint64)
    pts.tofile(tmp_path / "p.bin")
    send.tofile(tmp_path / "s.bin")
    subprocess.check_call([exe, "msm", str(tmp_path / "p.bin"), str(tmp_path / "s.bin"), str(n), str(mont), str(tmp_path / "o.bin")])
    got = np.fromfile(tmp_path / "o.bin", dtype=np.uint64)
    ref = pts[:, :12].copy()
    ref[5] = 0
    want = oracle.msm("bls12_381", ref, sc, "pippenger", ncpus=8)
    assert np.array_equal(oracle.jac_to_affine("bls12_381", got), oracle.jac_to_affine("bls12_381", want))


@pytest.mark.gpu
def test_cpp_example_preloaded_points(oracle, tmp_path):
    """msm_t{points, npoints}.invoke(out, scalars): the SRS stays on the GPU between invocations."""
    exe, _ = _builder().build_example()
    n = 4000
    pts = np.zeros((n, 13), dtype=np.uint64)
    pts[:, :12] = oracle.gen_points("bls12_381", 128)[np.arange(n) % 128]
    sc = _scalars(n, 77)
    pts.tofile(tmp_path / "p.bin")
    sc.tofile(tmp_path / "s.bin")
    subprocess.check_call([exe, "ctx", str(tmp_path / "p.bin"), str(tmp_path / "s.bin"), str(n), "0", str(tmp_path / "o.bin")])
    got = np.fromfile(tmp_path / "o.bin", dtype=np.uint64).reshape(2, 18)
    flat = np.ascontiguousarray(pts[:, :12])
    for k, m in enumerate((n, n // 2)):
        want = oracle.msm("bls12_381", flat[:m], sc[:m], "pippenger", ncpus=8)
        assert np.array_equal(oracle.jac_to_affine("bls12_381", got[k]), oracle.jac_to_affine("bls12_381", want)), m


@pytest.mark.gpu
def test_cpp_example_ntt(oracle, tmp_path):
    _, exe = _builder().build_example()
    rng = np.random.default_rng(3)
    x = rng.integers(0, GL_P, size=1 << 12, dtype=np.uint64)
    x.tofile(tmp_path / "d.bin")
    subprocess.check_call([exe, "ntt", str(tmp_path / "d.bin"), "12", "0", "0", "1"])      # NN, forward, coset
    got = np.fromfile(tmp_path / "d.bin", dtype=np.uint64)
    assert np.array_equal(got, oracle.ntt_gl64(x, oracle.NN, False, True))


@pytest.mark.gpu
def test_reference_poc_glue_runs_on_this_library(oracle):
    """The entry points DEFINED BY THE REFERENCE'S OWN .cu glue (compiled in the authoring container
    against include/compat, shipped as tests/cpp/_build/libdropin_*.so) give the oracle's answers."""
    path = os.path.join(OUT, "libdropin_msm.so")
    if not os.path.exists(path):
        pytest.skip("needs the glue libraries built from the original project's poc sources, which cannot be part of this repository")
    glue = C.CDLL(path)
    for f in (glue.mult_pippenger_inf, glue.mult_pippenger_fp2_inf):
        f.restype, f.argtypes = RE, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]
    n = 2000
    sc = _scalars(n, 8)
    pts = np.zeros((n, 13), dtype=np.uint64)
    pts[:, :12] = oracle.gen_points("bls12_381", 100)[np.arange(n) % 100]
    out = np.zeros(18, dtype=np.uint64)
    assert glue.mult_pippenger_inf(out.ctypes.data, pts.ctypes.data, n, sc.ctypes.data, 104).code == 0
    want = oracle.msm("bls12_381", np.ascontiguousarray(pts[:, :12]), sc, "pippenger", ncpus=8)
    assert np.array_equal(oracle.jac_to_affine("bls12_381", out), oracle.jac_to_affine("bls12_381", want))
    p2 = np.zeros((n, 25), dtype=np.uint64)
    p2[:, :24] = oracle.g2_points(100)[np.arange(n) % 100]
    out2 = np.zeros(36, dtype=np.uint64)
    assert glue.mult_pippenger_fp2_inf(out2.ctypes.data, p2.ctypes.data, n, sc.ctypes.data, 200).code == 0
    assert np.array_equal(oracle.g2_jac_to_affine(out2), oracle.g2_jac_to_affine(oracle.g2_msm(p2, sc)))
    g1 = C.CDLL(os.path.join(OUT, "libdropin_msm_g1.so"))
    g1.mult_pippenger.restype, g1.mult_pippenger.argtypes = RE, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    flat = np.ascontiguousarray(pts[:, :12])
    assert g1.mult_pippenger(out.ctypes.data, flat.ctypes.data, n, sc.ctypes.data).code == 0
    assert np.array_equal(oracle.jac_to_affine("bls12_381", out), oracle.jac_to_affine("bls12_381", want))
    for curve, lib, fr in (("bn254", "libdropin_msm_bn254.so", "bn254_fr"), ("bls12_377", "libdropin_msm_bls12_377.so", "bls12_377_fr")):
        glue = C.CDLL(os.path.join(OUT, lib))                # pippenger_inf.cu built with FEATURE_BN254 / _BLS12_377
        glue.mult_pippenger_inf.restype = RE
        glue.mult_pippenger_inf.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]
        nl = oracle.CURVE_LIMBS[oracle.CURVES[curve]]
        rmod = oracle.ff_consts(fr)["p"]
        rnd = random.Random(nl)
        sc2 = np.array([_limbs(rnd.randrange(rmod)) for _ in range(500)], dtype=np.uint64)
        ark = np.zeros((500, 2 * nl + 1), dtype=np.uint64)
        ark[:, :2 * nl] = oracle.gen_points(curve, 50)[np.arange(500) % 50]
        o2 = np.zeros(3 * nl, dtype=np.uint64)
        assert glue.mult_pippenger_inf(o2.ctypes.data, ark.ctypes.data, 500, sc2.ctypes.data, ark.strides[0]).code == 0
        w2 = oracle.msm(curve, np.ascontiguousarray(ark[:, :2 * nl]), sc2, "pippenger", ncpus=8)
        assert np.array_equal(oracle.jac_to_affine(curve, o2), oracle.jac_to_affine(curve, w2)), curve
        # the same glue's G2 entry (pippenger_inf.cu:36-47 over that feature's fp2_t), arkworks G2Affine rows
        from oracle import g2py
        c = g2py.curve(curve + "_g2")
        glue.mult_pippenger_fp2_inf.restype = RE
        glue.mult_pippenger_fp2_inf.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]
        base = g2py.multiples(c, 16)
        idx = [rnd.randrange(16) for _ in range(60)]
        g2rows = np.zeros((60, 4 * c.nl + 1), dtype=np.uint64)
        g2rows[:, :4 * c.nl] = c.encode_affine([base[i] for i in idx])
        g2rows[7, 4 * c.nl] = 1                              # flagged infinity
        o3 = np.zeros(6 * c.nl, dtype=np.uint64)
        assert glue.mult_pippenger_fp2_inf(o3.ctypes.data, g2rows.ctypes.data, 60, sc2.ctypes.data, g2rows.strides[0]).code == 0
        ks = [int(sum(int(v) << (64 * j) for j, v in enumerate(row))) for row in sc2[:60]]
        pts = [None if i == 7 else base[idx[i]] for i in range(60)]
        assert c.jacobian_to_affine(o3) == c.msm(pts, ks), curve + " G2 through the reference's glue"
    rng = np.random.default_rng(5)
    for lib, dt, p, ofn in (("libdropin_ntt_gl64.so", np.uint64, GL_P, oracle.ntt_gl64),
                            ("libdropin_ntt_bb31.so", np.uint32, 0x78000001, oracle.ntt_bb31)):
        ntt = C.CDLL(os.path.join(OUT, lib))
        ntt.compute_ntt.restype = RE
        ntt.compute_ntt.argtypes = [C.c_size_t, C.c_void_p, C.c_uint32, C.c_int, C.c_int, C.c_int]
        x = rng.integers(0, p, size=1 << 13, dtype=dt)
        for order, inv in ((0, 0), (1, 0), (2, 1)):
            y = x.copy()
            assert ntt.compute_ntt(0, y.ctypes.data, 13, order, inv, 0).code == 0
            assert np.array_equal(y, ofn(x, order, bool(inv))), (lib, order, inv)
    ntt = C.CDLL(os.path.join(OUT, "libdropin_ntt_bls12_381.so"))
    ntt.compute_ntt.restype = RE
    ntt.compute_ntt.argtypes = [C.c_size_t, C.c_void_p, C.c_uint32, C.c_int, C.c_int, C.c_int]
    x = rng.integers(0, 2**62, size=(1 << 10, 4), dtype=np.uint64)
    y = x.copy()
    assert ntt.compute_ntt(0, y.ctypes.data, 10, 0, 0, 0).code == 0
    assert np.array_equal(y, oracle.ntt_ff("bls12_381_fr", x, oracle.NN))

"""Generates the committed golden vectors from THE REFERENCE ITSELF (not from the oracle):

  ntt_ref_gpu.npz   inputs/outputs of the reference's own CUDA NTT (poc/ntt-cuda/cuda/ntt_api.cu
                    compiled for sm_100a into oracle/_ref by oracle/Makefile), Goldilocks and
                    BabyBear, lg 1..10, every order x direction x type.  Needs a GPU: run as
                    `gpurun -- python tests/golden/make_golden.py gpu` and copy gpurun_out/golden/*.
  msm_ref_gpu.npz   same for the reference's CUDA mult_pippenger (BLS12-381 G1).
  msm_g2_ref_gpu.npz  the reference's mult_pippenger_fp2_inf (BLS12-381 G2) and mult_pippenger_inf
                    (G1, arkworks layout with infinity flags): `... make_golden.py g2` on a GPU.
  msm_curves2_ref_gpu.npz  the reference's CUDA MSM for BN254 and BLS12-377 G1: `... make_golden.py curves2`.
  msm_pasta_ref_gpu.npz    the reference's CUDA MSM templates for Pallas and Vesta: `... make_golden.py pasta`.
  msm_g2_<curve>_ref_gpu.npz  the reference's CUDA MSM over Fp2 for BN254 and BLS12-377 (G2):
                    `... make_golden.py g2_bn254|g2_bls12_377`.
  poly_<field>_ref_gpu.npz  the reference's polynomial/ templates (prefix_op, div_by_x_minus_z,
                    evaluate) through oracle/ref_poly.cu: `... make_golden.py poly_gl64|poly_bb31|poly_bls12_381_fr`.
  msm_ref_cpu.npz, msm_ref_cpu_n700.npz   the reference's CPU msm/pippenger.hpp
                    (oracle/_ref/libref_msm_cpu.so); runs anywhere: `python tests/golden/make_golden.py cpu`.
  msm_ref_gpu_2pow26.npz  the reference's CUDA mult_pippenger on the 2^26-point input of
                    tests/test_msm_gpu.py: `... make_golden.py msm_2pow26` on a GPU.
  ref_params.json   the parameter tables of the reference's headers, read from a checkout of it:
                    `python tests/golden/make_golden.py params <reference checkout>`.

tests/test_oracle.py checks the CPU oracle against all three, which is what pins it.
Inputs are seeded; nothing here reads /root/reference at run time (only the prebuilt _ref .so).
"""
import ctypes as C
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import pyoracle as o  # noqa: E402

GL_P = 2**64 - 2**32 + 1
BB_P = 0x78000001
R_BLS = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001


class RE(C.Structure):
    _fields_ = [("code", C.c_int), ("message", C.c_void_p)]


def ok(e, what=""):
    if e.code != 0:
        msg = C.cast(e.message, C.c_char_p).value if e.message else b""
        raise RuntimeError(f"{what}: reference returned {e.code}: {msg.decode(errors='replace')}")


def msm_inputs():
    """A few small deterministic MSM instances (points = multiples of G, incl. infinity)."""
    rng = np.random.default_rng(2024)
    base = o.gen_points("bls12_381", 64)
    cases = {}
    for n in (1, 2, 33, 200, 1000):
        pts = base[np.arange(n) % 64].copy()
        if n > 3:
            pts[3] = 0
        sc = rng.integers(0, 2**64, size=(n, 4), dtype=np.uint64)
        sc[:, 3] >>= np.uint64(2)
        if n >= 33:
            sc[5] = 0
            sc[6] = [1, 0, 0, 0]
            sc[7] = o.int_to_limbs(R_BLS - 1, 4)
        cases[n] = (pts, sc)
    return cases


def gen_cpu(outdir):
    cases = msm_inputs()
    out = {}
    for n, (pts, sc) in cases.items():
        jac = o.ref_cpu_msm(pts, sc, nthreads=4)
        out[f"pts_{n}"] = pts
        out[f"sc_{n}"] = sc
        out[f"affine_{n}"] = o.jac_to_affine("bls12_381", jac)
    np.savez_compressed(os.path.join(outdir, "msm_ref_cpu.npz"), **out)
    print("wrote msm_ref_cpu.npz")
    # 700 points: 50 distinct multiples of G, scalars uniform below r (random.Random(3))
    import random
    rnd = random.Random(3)
    n = 700
    pts = o.gen_points("bls12_381", 50)[np.arange(n) % 50].copy()
    sc = np.array([o.int_to_limbs(rnd.randrange(R_BLS), 4) for _ in range(n)], dtype=np.uint64)
    affine = o.jac_to_affine("bls12_381", o.ref_cpu_msm(pts, sc, nthreads=4))
    np.savez_compressed(os.path.join(outdir, "msm_ref_cpu_n700.npz"), pts=pts, sc=sc, affine=affine)
    print("wrote msm_ref_cpu_n700.npz")


# Every reference library is loaded in a process of its own: the reference's NTT keeps its
# parameter tables in function-local / template statics, which g++ emits as STB_GNU_UNIQUE symbols;
# the dynamic loader then shares ONE copy between all libraries of a process even under
# RTLD_LOCAL, so a BabyBear library loaded after the Goldilocks one computes with Goldilocks
# tables (this is what made the round-1 BabyBear / 256-bit recordings look self-inconsistent).
def gen_ntt_word(outdir, field):
    dtype, p, so = {"gl64": (np.uint64, GL_P, "libref_ntt_gl64_gpu.so"),
                    "bb31": (np.uint32, BB_P, "libref_ntt_bb31_gpu.so")}[field]
    out = {}
    lib = C.CDLL(o.ref_path(so))
    lib.compute_ntt.restype = RE
    lib.compute_ntt.argtypes = [C.c_size_t, C.c_void_p, C.c_uint32, C.c_int, C.c_int, C.c_int]
    rng = np.random.default_rng(7 if field == "gl64" else 8)
    for lg in range(1, 13 if field == "bb31" else 11):
        x = rng.integers(0, p, size=1 << lg, dtype=dtype)
        out[f"{field}_in_{lg}"] = x
        for order in range(4):
            for direction in range(2):
                for typ in range(2):
                    y = x.copy()
                    e = lib.compute_ntt(0, y.ctypes.data, lg, order, direction, typ)
                    assert e.code == 0
                    out[f"{field}_out_{lg}_{order}{direction}{typ}"] = y
    np.savez_compressed(os.path.join(outdir, f"ntt_{field}_ref_gpu.npz"), **out)
    print(f"wrote ntt_{field}_ref_gpu.npz")


def gen_lde(outdir):
    # low-degree extension, Goldilocks (NTT::LDE)
    lib = C.CDLL(o.ref_path("libref_ntt_gl64_gpu.so"))
    lib.ref_lde.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32]
    rng = np.random.default_rng(21)
    out = {}
    for lg, lb in ((1, 1), (3, 1), (6, 2), (10, 1), (12, 3)):
        x = rng.integers(0, GL_P, size=1 << lg, dtype=np.uint64)
        buf = np.zeros(1 << (lg + lb), dtype=np.uint64)
        buf[: 1 << lg] = x
        assert lib.ref_lde(buf.ctypes.data, lg, lb) == 0
        out[f"in_{lg}_{lb}"] = x
        out[f"out_{lg}_{lb}"] = buf
    np.savez_compressed(os.path.join(outdir, "lde_ref_gpu.npz"), **out)
    print("wrote lde_ref_gpu.npz")


def gen_ntt256(outdir):
    # 256-bit "wide" NTT: BLS12-381 scalar field, Montgomery residues
    lib = C.CDLL(o.ref_path("libref_ntt_bls12_381_gpu.so"))
    lib.compute_ntt.restype = RE
    lib.compute_ntt.argtypes = [C.c_size_t, C.c_void_p, C.c_uint32, C.c_int, C.c_int, C.c_int]
    out = {}
    for lg, x in o.ntt256_inputs().items():
        for order in range(4):
            for direction in range(2):
                for typ in range(2):
                    y = x.copy()
                    e = lib.compute_ntt(0, y.ctypes.data, lg, order, direction, typ)
                    assert e.code == 0
                    out[f"out_{lg}_{order}{direction}{typ}"] = y
        # not stored, restored by oracle.pyoracle.ntt256_golden: the input (ntt256_inputs) and the
        # RR outputs of the plain transforms, equal to the NN ones
        for direction in range(2):
            assert np.array_equal(out.pop(f"out_{lg}_3{direction}0"), out[f"out_{lg}_0{direction}0"])
    np.savez_compressed(os.path.join(outdir, "ntt256_ref_gpu.npz"), **out)
    print("wrote ntt256_ref_gpu.npz")


def gen_msm(outdir):
    lib = C.CDLL(o.ref_path("libref_msm_gpu.so"))
    lib.mult_pippenger.restype = RE
    lib.mult_pippenger.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    out = {}
    for n, (pts, sc) in msm_inputs().items():
        jac = np.zeros(18, dtype=np.uint64)
        e = lib.mult_pippenger(jac.ctypes.data, pts.ctypes.data, n, sc.ctypes.data)
        assert e.code == 0
        out[f"pts_{n}"] = pts
        out[f"sc_{n}"] = sc
        out[f"affine_{n}"] = o.jac_to_affine("bls12_381", jac)
    np.savez_compressed(os.path.join(outdir, "msm_ref_gpu.npz"), **out)
    print("wrote msm_ref_gpu.npz")


def gen_msm_2pow26(outdir):
    """msm_ref_gpu_2pow26.npz: the reference's CUDA mult_pippenger on 2^26 points, the 2^16
    multiples (i+1)*G replicated, scalars uniform below 2^254 from default_rng(26) in blocks of
    2^22 rows -- the input of tests/test_msm_gpu.py::test_bls12_381_msm_2pow26_equals_reference_gpu."""
    lib = C.CDLL(o.ref_path("libref_msm_gpu.so"))
    lib.mult_pippenger.restype = RE
    lib.mult_pippenger.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    n, m = 1 << 26, 1 << 16
    pts = np.empty((n, 12), dtype=np.uint64)
    pts.reshape(n // m, m, 12)[:] = o.gen_points("bls12_381", m)
    rng = np.random.default_rng(26)
    sc = np.empty((n, 4), dtype=np.uint64)
    for s in range(0, n, 1 << 22):
        sc[s:s + (1 << 22)] = rng.integers(0, 2**64, size=(1 << 22, 4), dtype=np.uint64)
    sc[:, 3] >>= np.uint64(2)
    jac = np.zeros(18, dtype=np.uint64)
    ok(lib.mult_pippenger(jac.ctypes.data, pts.ctypes.data, n, sc.ctypes.data), "mult_pippenger 2^26")
    np.savez_compressed(os.path.join(outdir, "msm_ref_gpu_2pow26.npz"), out=jac)
    print("wrote msm_ref_gpu_2pow26.npz")


def gen_gpu(outdir):
    """all GPU goldens, one process per reference library; ntt_ref_gpu.npz = Goldilocks + BabyBear"""
    import subprocess
    for mode in ("ntt_gl64", "ntt_bb31", "lde", "ntt256", "msm"):
        subprocess.check_call([sys.executable, os.path.abspath(__file__), mode])
    merged = {}
    for field in ("gl64", "bb31"):
        part = os.path.join(outdir, f"ntt_{field}_ref_gpu.npz")
        with np.load(part) as g:
            merged.update({k: g[k] for k in g.files})
        os.remove(part)
    np.savez_compressed(os.path.join(outdir, "ntt_ref_gpu.npz"), **merged)
    print("wrote ntt_ref_gpu.npz")


def g2_inputs():
    """Small deterministic G2 instances in the arkworks layout (n, 25): X, Y in Fp2 + flag word."""
    rng = np.random.default_rng(381)
    base = o.g2_points(64)
    cases = []
    for n in (1, 2, 33, 200, 1000):
        pts = np.zeros((n, 25), dtype=np.uint64)
        pts[:, :24] = base[rng.integers(0, 64, size=n)]
        if n > 3:
            pts[3, 24] = 1                       # flagged infinity
        sc = rng.integers(0, 2**64, size=(n, 4), dtype=np.uint64)
        sc[:, 3] >>= np.uint64(2)
        if n >= 33:
            sc[5] = 0
            sc[6] = [1, 0, 0, 0]
            sc[7] = o.int_to_limbs(R_BLS - 1, 4)
            pts[9] = pts[8]                      # equal points, equal scalars -> doubling in a bucket
            sc[9] = sc[8]
        cases.append((pts, sc))
    return cases


def gen_g2(outdir):
    """msm_g2_ref_gpu.npz: the reference's mult_pippenger_fp2_inf (and, for the G1 arkworks layout,
    mult_pippenger_inf) from oracle/_ref/libref_msm_g2_gpu.so, run on a B200."""
    lib = C.CDLL(o.ref_path("libref_msm_g2_gpu.so"))
    for f in (lib.mult_pippenger_fp2_inf, lib.mult_pippenger_inf):
        f.restype = RE
        f.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]
    packed = C.CDLL(o.ref_path("libref_msm_g2_packed_gpu.so"))
    packed.ref_mult_pippenger_fp2.restype = RE
    packed.ref_mult_pippenger_fp2.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    out = {}
    cases = g2_inputs()
    for k, (pts, sc) in enumerate(cases):
        # out{k}: the reference's templates on packed points (flagged rows -> X = Y = 0), the pin.
        # inf_out{k}: the reference's mult_pippenger_fp2_inf as built -- kept as evidence of its
        # host/device layout mismatch (oracle/ref_msm_g2.cu), not used as an expectation.
        flat = np.ascontiguousarray(pts[:, :24])
        flat[pts[:, 24] != 0] = 0
        jac = np.zeros(36, dtype=np.uint64)
        e = packed.ref_mult_pippenger_fp2(jac.ctypes.data, flat.ctypes.data, flat.shape[0], sc.ctypes.data)
        ok(e, f"packed fp2 n={flat.shape[0]}")
        inf = np.zeros(36, dtype=np.uint64)
        e = lib.mult_pippenger_fp2_inf(inf.ctypes.data, pts.ctypes.data, pts.shape[0], sc.ctypes.data, 200)
        ok(e, f"fp2_inf n={pts.shape[0]}")
        out[f"points{k}"], out[f"scalars{k}"], out[f"out{k}"], out[f"inf_out{k}"] = pts, sc, jac, inf
    out["ncases"] = np.int64(len(cases))
    g1 = 0
    for n, (pts, sc) in msm_inputs().items():
        ark = np.zeros((n, 13), dtype=np.uint64)
        ark[:, :12] = pts
        if n > 10:
            ark[10, 12] = 1
        jac = np.zeros(18, dtype=np.uint64)
        e = lib.mult_pippenger_inf(jac.ctypes.data, ark.ctypes.data, n, sc.ctypes.data, 104)
        assert e.code == 0
        out[f"g1_points{g1}"], out[f"g1_scalars{g1}"], out[f"g1_out{g1}"] = ark, sc, jac
        g1 += 1
    out["g1_ncases"] = np.int64(g1)
    np.savez_compressed(os.path.join(outdir, "msm_g2_ref_gpu.npz"), **out)
    print("wrote msm_g2_ref_gpu.npz")


def gen_curves2(outdir):
    """msm_curves2_ref_gpu.npz: the reference's CUDA MSM templates for the msm crate's bn254 and
    bls12_377 features (oracle/ref_msm_g1.cu -> mult_pippenger_inf, arkworks rows with flags)."""
    out = {}
    for curve, lib, r in (("bn254", "libref_msm_bn254_gpu.so", 0x30644e72e131a029b85045b68181585d2833e84879b9709143e1f593f0000001),
                          ("bls12_377", "libref_msm_bls12_377_gpu.so", 0x12ab655e9a2ca55660b44d1e5c37b00159aa76fed00000010a11800000000001)):
        ref = C.CDLL(o.ref_path(lib))
        ref.mult_pippenger_inf.restype = RE
        ref.mult_pippenger_inf.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]
        nl = o.CURVE_LIMBS[o.CURVES[curve]]
        rng = np.random.default_rng(nl)
        base = o.gen_points(curve, 64)
        k = 0
        for n in (1, 2, 33, 200, 1000):
            pts = np.zeros((n, 2 * nl + 1), dtype=np.uint64)
            pts[:, :2 * nl] = base[rng.integers(0, 64, size=n)]
            sc = np.array([o.int_to_limbs(int.from_bytes(rng.bytes(32), "little") % r, 4) for _ in range(n)], dtype=np.uint64)
            if n > 10:
                pts[3, 2 * nl] = 1
                pts[4, :2 * nl] = 0
                sc[5] = 0
                sc[7] = o.int_to_limbs(r - 1, 4)
                pts[9], sc[9] = pts[8], sc[8]
            jac = np.zeros(3 * nl, dtype=np.uint64)
            ok(ref.mult_pippenger_inf(jac.ctypes.data, pts.ctypes.data, n, sc.ctypes.data, pts.strides[0]), f"{curve} n={n}")
            out[f"{curve}_points{k}"], out[f"{curve}_scalars{k}"], out[f"{curve}_out{k}"] = pts, sc, jac
            k += 1
        out[f"{curve}_ncases"] = np.int64(k)
    np.savez_compressed(os.path.join(outdir, "msm_curves2_ref_gpu.npz"), **out)
    print("wrote msm_curves2_ref_gpu.npz")


def gen_pasta(outdir):
    """msm_pasta_ref_gpu.npz: the reference's CUDA MSM templates instantiated for the Pasta curves
    (oracle/ref_msm_g1.cu with FEATURE_PALLAS / FEATURE_VESTA over ff/pasta.hpp; host field types from
    oracle/shim/pasta_t.hpp): rows x, y, infinity flag; scalars are integers below the group order."""
    out = {}
    orders = {"pallas": 0x40000000000000000000000000000000224698fc0994a8dd8c46eb2100000001,
              "vesta": 0x40000000000000000000000000000000224698fc094cf91b992d30ed00000001}
    for curve, lib in (("pallas", "libref_msm_pallas_gpu.so"), ("vesta", "libref_msm_vesta_gpu.so")):
        r = orders[curve]
        ref = C.CDLL(o.ref_path(lib))
        ref.mult_pippenger_inf.restype = RE
        ref.mult_pippenger_inf.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]
        nl = o.CURVE_LIMBS[o.CURVES[curve]]
        rng = np.random.default_rng(100 + nl)
        base = o.gen_points(curve, 64)
        k = 0
        for n in (1, 2, 33, 200, 1000, 5000):
            pts = np.zeros((n, 2 * nl + 1), dtype=np.uint64)
            pts[:, :2 * nl] = base[rng.integers(0, 64, size=n)]
            sc = np.array([o.int_to_limbs(int.from_bytes(rng.bytes(32), "little") % r, 4) for _ in range(n)], dtype=np.uint64)
            if n > 10:
                pts[3, 2 * nl] = 1
                pts[4, :2 * nl] = 0
                sc[5] = 0
                sc[7] = o.int_to_limbs(r - 1, 4)
                pts[9], sc[9] = pts[8], sc[8]
            jac = np.zeros(3 * nl, dtype=np.uint64)
            ok(ref.mult_pippenger_inf(jac.ctypes.data, pts.ctypes.data, n, sc.ctypes.data, pts.strides[0]), f"{curve} n={n}")
            out[f"{curve}_points{k}"], out[f"{curve}_scalars{k}"], out[f"{curve}_out{k}"] = pts, sc, jac
            k += 1
        out[f"{curve}_ncases"] = np.int64(k)
    np.savez_compressed(os.path.join(outdir, "msm_pasta_ref_gpu.npz"), **out)
    print("wrote msm_pasta_ref_gpu.npz")


def gen_poly(outdir, field):
    """poly_<field>_ref_gpu.npz: the reference's polynomial/ templates (oracle/ref_poly.cu) on
    seeded inputs in the field's memory format.  One reference library per process.  Two limits
    of the reference itself are stepped around (profiles/ref_poly_probe_r02.txt): its evaluate
    faults at len = 1, and its 256-bit div_by_x_minus_z faults for len <= 5001 -- those cases are
    not recorded.  The `big` case keeps SHA-256 digests of the outputs instead of the arrays; its
    input is regenerated from the seed by oracle.poly.seeded_input."""
    import hashlib
    from oracle import poly as op
    lib = C.CDLL(o.ref_path(f"libref_poly_{field if field != 'bls12_381_fr' else 'bls12_381'}_gpu.so"))
    lib.ref_prefix_op.argtypes = [C.c_int, C.c_void_p, C.c_size_t]
    lib.ref_div_by_x_minus_z.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_int]
    lib.ref_evaluate.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]
    f = op.FIELDS[field]
    wide = f["words"] > 1
    assert lib.ref_poly_elem_bytes() == f["words"] * np.dtype(f["dtype"]).itemsize
    import random
    rnd = random.Random({"gl64": 1, "bb31": 2, "bls12_381_fr": 3}[field])
    lens = (1, 2, 33, 255, 1024, 1025, 3000, 5001) if wide else \
           (1, 2, 3, 31, 32, 33, 255, 1000, 2048, 2049, 10000, 20001)
    big = 65536 if wide else (1 << 20) + 1
    out = {"lens": np.array(lens, dtype=np.int64), "big": np.int64(big)}

    def call(e, what):
        if e != 0:
            raise RuntimeError(f"reference {what}: cuda error {e}")

    for n in lens + (big,):
        digest = n == big
        if digest:
            x = op.seeded_input(field, n, 4242)
            vals = None
        else:
            vals = [rnd.randrange(f["p"]) for _ in range(n)]
            if n > 40:
                vals[7] = 0
                vals[n - 2] = f["p"] - 1
            x = op.encode(field, vals)
            out[f"in_{n}"] = x

        def keep(key, y):
            out[key] = np.frombuffer(hashlib.sha256(y.tobytes()).digest(), dtype=np.uint8) if digest else y

        for name, opc in (("add", 0), ("mul", 1)):
            y = x.copy()
            if name == "mul" and n > 40 and not digest:       # keep the products non-zero past index 7
                y[7] = op.encode(field, [3])[0]
                out[f"mulin_{n}"] = y.copy()
            call(lib.ref_prefix_op(opc, y.ctypes.data, n), f"prefix_op {name} {n}")
            keep(f"{name}_{n}", y)
        zs = [rnd.randrange(f["p"])]
        if n in (33, 1000, 1024):
            zs += [0, 1]
        out[f"z_{n}"] = op.encode(field, zs)
        if not wide or digest:
            for k, z in enumerate(zs):
                zbuf = op.encode(field, [z])
                for rot in (0, 1):
                    y = x.copy()
                    call(lib.ref_div_by_x_minus_z(y.ctypes.data, n, zbuf.ctypes.data, rot), f"div {n} {rot}")
                    keep(f"div_{n}_{k}_{rot}", y)
        if n > 1:
            npts = {33: 3, 1000: 7, 1024: 7}.get(n, 2)
            xs = op.encode(field, [rnd.randrange(f["p"]) for _ in range(npts - 1)] + [0])
            ret = np.zeros_like(xs)
            call(lib.ref_evaluate(ret.ctypes.data, xs.ctypes.data, npts, x.ctypes.data, n), f"evaluate {n}")
            out[f"x_{n}"], out[f"eval_{n}"] = xs, ret
    np.savez_compressed(os.path.join(outdir, f"poly_{field}_ref_gpu.npz"), **out)
    print(f"wrote poly_{field}_ref_gpu.npz")


def gen_params(outdir, ref):
    """ref_params.json: the parameter tables the reference hard-codes in its headers (roots of
    unity, domain-size inverses, Montgomery constants), read from the reference checkout `ref`,
    as hex strings (tests/test_params_pin.py compares the derived values with them)."""
    import json
    import re

    def small_table(path, name):
        s = open(path).read()
        tail = s.split("#endif")[-1]
        if "#else" in s:
            s = s.split("#else")[1].split("#endif")[0]
        m = re.search(r"const fr_t %s\[S \+ 1\] = \{(.*?)\};" % name, s + tail, re.S)
        return [int(x, 16) for x in re.findall(r"fr_t\((0x[0-9a-f]+)u?\)", m.group(1))]

    def words(path, name):
        """32-bit words of a device-side constant of ff/*.hpp"""
        s = open(path).read().split("namespace device")[1]
        m = re.search(r"%s\[\d+\] = \{(.*?)\};" % name, s, re.S)
        w = []
        for v in re.findall(r"TO_CUDA_T\((0x[0-9a-f]+)\)", m.group(1)):
            v = int(v, 16)
            w += [v & 0xFFFFFFFF, v >> 32]
        if not w:                                       # pasta.hpp lists plain 32-bit words
            w = [int(v, 16) for v in re.findall(r"0x[0-9a-f]{8}", m.group(1))]
        return w

    def wide_tables(path):
        s = open(path).read()
        t = {}
        for m in re.finditer(r"const fr_t (\w+)\[S \+ 1\] = \{(.*?)\};", s, re.S):
            vals = []
            for mm in re.finditer(r"FR_T\(vec256,(.*?)\)", m.group(2)):
                l = [int(x.strip().rstrip("u"), 16) for x in mm.group(1).split(",")]
                vals.append(sum(v << (64 * i) for i, v in enumerate(l)))
            t[m.group(1)] = vals
        m = re.search(r"const fr_t group_gen = FR_T\(vec256,(.*?)\)", s)
        l = [int(x.strip().rstrip("u"), 16) for x in m.group(1).split(",")]
        t["group_gen"] = [sum(v << (64 * i) for i, v in enumerate(l))]
        return {k: t[k] for k in ("group_gen", "forward_roots_of_unity", "domain_size_inverse")}

    out = {"ntt": {}, "ff": {}, "ntt256": {}}
    for name in ("goldilocks", "baby_bear"):
        out["ntt"][name] = {t: small_table(f"{ref}/ntt/parameters/{name}.h", t)
                            for t in ("forward_roots_of_unity", "inverse_roots_of_unity", "domain_size_inverse")}
    for hdr, names in (("bls12-381", ("BLS12_381_P", "BLS12_381_RR", "BLS12_381_one", "BLS12_381_r", "BLS12_381_rone")),
                       ("pasta", ("Pallas_P", "Pallas_RR", "Pallas_one", "Vesta_P", "Vesta_RR", "Vesta_one")),
                       ("alt_bn128", ("ALT_BN128_P", "ALT_BN128_RR", "ALT_BN128_one", "ALT_BN128_r", "ALT_BN128_rRR",
                                      "ALT_BN128_rone")),
                       ("bls12-377", ("BLS12_377_P", "BLS12_377_RR", "BLS12_377_one", "BLS12_377_r", "BLS12_377_rone"))):
        out["ff"][hdr] = {n: words(f"{ref}/ff/{hdr}.hpp", n) for n in names}
    for name in ("bls12_381", "vesta", "pallas", "alt_bn128", "bls12_377"):
        out["ntt256"][name] = wide_tables(f"{ref}/ntt/parameters/{name}.h")
    hexed = {sec: {k: {t: [hex(v) for v in vs] for t, vs in d.items()} for k, d in tab.items()} for sec, tab in out.items()}
    with open(os.path.join(outdir, "ref_params.json"), "w") as f:
        json.dump(hexed, f, indent=1)
        f.write("\n")
    print("wrote ref_params.json")


def gen_g2_curve(outdir, name):
    """msm_g2_<curve>_ref_gpu.npz: the reference's CUDA MSM templates over Fp2 for the msm crate's
    bn254 / bls12_377 features (oracle/ref_msm_g2.cu built with FEATURE_BN254 / FEATURE_BLS12_377:
    packed affine rows, see that file for why not mult_pippenger_fp2_inf itself).  Points are
    multiples of an order-r point (oracle/g2py.py), so every scalar below r is legitimate."""
    import random
    from oracle import g2py
    c = g2py.curve(name + "_g2")
    ref = C.CDLL(o.ref_path(f"libref_msm_g2_packed_{name}_gpu.so"))
    ref.ref_mult_pippenger_fp2.restype = RE
    ref.ref_mult_pippenger_fp2.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    rnd = random.Random(c.nl)
    base = g2py.multiples(c, 64)
    out, k = {}, 0
    for n in (1, 2, 33, 200, 1000):
        pts = [base[rnd.randrange(64)] for _ in range(n)]
        sc = [rnd.randrange(c.r) for _ in range(n)]
        if n > 10:
            pts[3] = None                                   # infinity row (all zero)
            sc[5], sc[6], sc[7] = 0, 1, c.r - 1
            pts[9], sc[9] = pts[8], sc[8]                   # the same term twice
            pts[11] = c.neg(pts[10])                        # P and -P in one bucket
            sc[11] = sc[10]
        rows, srows = c.encode_affine(pts), g2py.scalars_to_rows(sc)
        jac = np.zeros(6 * c.nl, dtype=np.uint64)
        ok(ref.ref_mult_pippenger_fp2(jac.ctypes.data, rows.ctypes.data, n, srows.ctypes.data), f"{name} g2 n={n}")
        out[f"points{k}"], out[f"scalars{k}"], out[f"out{k}"] = rows, srows, jac
        k += 1
    out["ncases"] = np.int64(k)
    np.savez_compressed(os.path.join(outdir, f"msm_g2_{name}_ref_gpu.npz"), **out)
    print(f"wrote msm_g2_{name}_ref_gpu.npz")


if __name__ == "__main__":
    mode = sys.argv[1] if len(sys.argv) > 1 else "cpu"
    if mode == "cpu":
        gen_cpu(HERE)
    elif mode == "params":
        gen_params(HERE, sys.argv[2])
    else:
        outdir = os.path.join(ROOT, "gpurun_out", "golden")
        os.makedirs(outdir, exist_ok=True)
        if mode == "g2":
            gen_g2(outdir)
        elif mode == "curves2":
            gen_curves2(outdir)
        elif mode == "pasta":
            gen_pasta(outdir)
        elif mode in ("ntt_gl64", "ntt_bb31"):
            gen_ntt_word(outdir, mode[4:])
        elif mode == "lde":
            gen_lde(outdir)
        elif mode == "ntt256":
            gen_ntt256(outdir)
        elif mode == "msm":
            gen_msm(outdir)
        elif mode == "msm_2pow26":
            gen_msm_2pow26(outdir)
        elif mode in ("g2_bn254", "g2_bls12_377"):
            gen_g2_curve(outdir, mode[3:])
        elif mode.startswith("poly_"):
            gen_poly(outdir, mode[5:])
        else:
            gen_gpu(outdir)

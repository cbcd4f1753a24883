"""ctypes binding of the CPU oracle -- TEST INFRASTRUCTURE ONLY.

liboracle.so   = the C restatement (oracle/ff.c ec.c ec2.c msm.c ntt.c)
_ref/*.so      = the reference's own sources compiled where they lie (oracle/Makefile),
                 present only if built in the authoring container.
All buffers are numpy arrays; field elements are little-endian 64-bit limbs.
"""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF_DIR = os.path.join(HERE, "_ref")

CURVES = {"bls12_381": 0, "pallas": 1, "vesta": 2, "bn254": 4, "bls12_377": 5}      # 3 = G2 (g2_* below)
FIELDS = {"bls12_381_fp": 0, "bls12_381_fr": 1, "pallas_fp": 2, "vesta_fp": 3,
          "bn254_fp": 4, "bn254_fr": 5, "bls12_377_fp": 6, "bls12_377_fr": 7}
FIELD_LIMBS = {0: 6, 1: 4, 2: 4, 3: 4, 4: 4, 5: 4, 6: 6, 7: 4}
CURVE_LIMBS = {0: 6, 1: 4, 2: 4, 4: 4, 5: 6}
NN, NR, RN, RR, BB = 0, 1, 2, 3, 4

_lib = None


def build(force=False):
    so = os.path.join(HERE, "liboracle.so")
    srcs = [os.path.join(HERE, f) for f in ("ff.c", "ec.c", "ec2.c", "msm.c", "ntt.c", "ff.h", "ec.h", "ec2.h", "msm.h", "ntt.h")]
    if force or not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.check_call(["make", "-s", "-C", HERE, "liboracle.so"])
    return so


def build_ref():
    """Compile the reference's own sources into oracle/_ref (authoring container only)."""
    if os.path.isdir("/root/reference"):
        subprocess.check_call(["make", "-s", "-C", HERE, "ref"])
        return True
    return False


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        _lib.oracle_msm.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t,
                                    C.c_void_p, C.c_int, C.c_int]
        _lib.oracle_points.argtypes = [C.c_int, C.c_void_p, C.c_size_t]
        _lib.oracle_jac_to_affine.argtypes = [C.c_int, C.c_void_p, C.c_void_p]
        _lib.oracle_affine_on_curve.argtypes = [C.c_int, C.c_void_p]
        _lib.oracle_ff_op.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        _lib.oracle_ff_consts.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        _lib.oracle_ntt_gl64.argtypes = [C.c_void_p, C.c_uint, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
        _lib.oracle_ntt_bb31.argtypes = [C.c_void_p, C.c_uint, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
        _lib.oracle_ntt_ff.argtypes = [C.c_int, C.c_void_p, C.c_uint, C.c_int, C.c_int, C.c_int, C.c_int]
        _lib.oracle_fp2_op.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        _lib.oracle_g2_points.argtypes = [C.c_void_p, C.c_size_t]
        _lib.oracle_g2_msm.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_size_t, C.c_void_p]
        _lib.oracle_g2_jac_to_affine.argtypes = [C.c_void_p, C.c_void_p]
        _lib.oracle_g2_on_curve.argtypes = [C.c_void_p]
        _lib.oracle_gl64_root.restype = C.c_uint64
        _lib.oracle_gl64_root.argtypes = [C.c_uint, C.c_int]
        _lib.oracle_bb31_root.restype = C.c_uint32
        _lib.oracle_bb31_root.argtypes = [C.c_uint, C.c_int]
    return _lib


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


# ---------------------------------------------------------------- integers <-> limbs
def int_to_limbs(x, n):
    return np.array([(x >> (64 * i)) & 0xFFFFFFFFFFFFFFFF for i in range(n)], dtype=np.uint64)


def limbs_to_int(a):
    return sum(int(v) << (64 * i) for i, v in enumerate(np.asarray(a, dtype=np.uint64).ravel()))


# ---------------------------------------------------------------- field
def ff_op(field, op, a, b=None):
    fid = FIELDS[field]
    n = FIELD_LIMBS[fid]
    opc = {"mul": 0, "add": 1, "sub": 2, "to_mont": 3, "from_mont": 4, "inv": 5}[op]
    r = np.zeros(n, dtype=np.uint64)
    aa = int_to_limbs(a, n)
    bb = int_to_limbs(b if b is not None else 0, n)
    lib().oracle_ff_op(fid, opc, _ptr(r), _ptr(aa), _ptr(bb))
    return limbs_to_int(r)


def ff_consts(field):
    fid = FIELDS[field]
    n = FIELD_LIMBS[fid]
    p, rr, one = (np.zeros(n, dtype=np.uint64) for _ in range(3))
    m0 = C.c_uint64(0)
    lib().oracle_ff_consts(fid, _ptr(p), C.byref(m0), _ptr(rr), _ptr(one))
    return dict(p=limbs_to_int(p), m0=m0.value, rr=limbs_to_int(rr), one=limbs_to_int(one), n=n)


# ---------------------------------------------------------------- curve / msm
def gen_points(curve, ndistinct):
    """(ndistinct, 2*n) uint64: affine (i+1)*G in Montgomery form."""
    cid = CURVES[curve]
    out = np.zeros((ndistinct, 2 * CURVE_LIMBS[cid]), dtype=np.uint64)
    lib().oracle_points(cid, _ptr(out), ndistinct)
    return out


def msm(curve, points, scalars, algo="pippenger", ncpus=1):
    """points: (n, >=2*limbs) uint64 rows (row stride taken from the array); scalars: (n,4) uint64.
    Returns jacobian (3*limbs,) uint64."""
    cid = CURVES[curve]
    nl = CURVE_LIMBS[cid]
    points = np.ascontiguousarray(points)
    scalars = np.ascontiguousarray(scalars, dtype=np.uint64)
    n = points.shape[0]
    assert scalars.shape[0] == n
    out = np.zeros(3 * nl, dtype=np.uint64)
    stride = points.strides[0] if n else 16 * nl
    lib().oracle_msm(cid, _ptr(out), _ptr(points), stride, n, _ptr(scalars), ncpus,
                     {"pippenger": 0, "serial": 1, "naive": 2}[algo])
    return out


def jac_to_affine(curve, jac):
    cid = CURVES[curve]
    out = np.zeros(2 * CURVE_LIMBS[cid], dtype=np.uint64)
    jac = np.ascontiguousarray(jac, dtype=np.uint64)
    lib().oracle_jac_to_affine(cid, _ptr(out), _ptr(jac))
    return out


def on_curve(curve, xy):
    xy = np.ascontiguousarray(xy, dtype=np.uint64)
    return bool(lib().oracle_affine_on_curve(CURVES[curve], _ptr(xy)))


# ---------------------------------------------------------------- ntt
def ntt_gl64(a, order=NN, inverse=False, coset=False, algo="fast", nthreads=1):
    a = np.array(a, dtype=np.uint64, copy=True)
    lg = int(a.size).bit_length() - 1
    assert a.size == 1 << lg
    rc = lib().oracle_ntt_gl64(_ptr(a), lg, order, int(inverse), int(coset), int(algo == "dft"), nthreads)
    assert rc == 0
    return a


def ntt_bb31(a, order=NN, inverse=False, coset=False, algo="fast", nthreads=1):
    a = np.array(a, dtype=np.uint32, copy=True)
    lg = int(a.size).bit_length() - 1
    assert a.size == 1 << lg
    rc = lib().oracle_ntt_bb31(_ptr(a), lg, order, int(inverse), int(coset), int(algo == "dft"), nthreads)
    assert rc == 0
    return a


def ntt_ff(field, a, order=NN, inverse=False, coset=False, algo="fast"):
    """256-bit fields: field in {'bls12_381_fr', 'pallas_fp', 'vesta_fp'}; a: (n, 4) uint64
    Montgomery residues."""
    a = np.array(a, dtype=np.uint64, copy=True).reshape(-1, 4)
    lg = int(a.shape[0]).bit_length() - 1
    assert a.shape[0] == 1 << lg
    rc = lib().oracle_ntt_ff(FIELDS[field], _ptr(a), lg, order, int(inverse), int(coset), int(algo == "dft"))
    assert rc == 0
    return a


def lde(field, evals, lg_blowup):
    """Definition of NTT::LDE (ntt/ntt.cuh:247-340): coefficients c = iNTT(evals); the extended
    array is the coset NTT, over the 2^(lg+lg_blowup) domain, of c padded with zeros."""
    fn = {"gl64": ntt_gl64, "bb31": ntt_bb31}.get(field) or (lambda a, *k, **kw: ntt_ff(field, a, *k, **kw))
    c = fn(evals, NN, True)
    ext = np.zeros((c.shape[0] << lg_blowup,) + c.shape[1:], dtype=c.dtype)
    ext[:c.shape[0]] = c
    return fn(ext, NN, False, True), c


def ntt256_inputs():
    """{lg: input} of the 256-bit NTT recording (tests/golden/make_golden.py ntt256), lg 1..10:
    BLS12-381 scalar-field residues, (2^lg, 4) uint64, drawn in turn from random.Random(11)."""
    import random
    r = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001
    rnd = random.Random(11)
    return {lg: np.array([int_to_limbs(rnd.randrange(r), 4) for _ in range(1 << lg)], dtype=np.uint64)
            for lg in range(1, 11)}


def ntt256_golden(path):
    """tests/golden/ntt256_ref_gpu.npz as a dict of every in_<lg> and
    out_<lg>_<order><direction><type>.  Two kinds of array are not stored: the inputs, which are
    ntt256_inputs(), and the RR outputs of the plain (non-coset) transforms, which the reference
    computes bit for bit equal to the NN ones (the file stays below 1 MB)."""
    g = dict(np.load(path))
    for lg, x in ntt256_inputs().items():
        g[f"in_{lg}"] = x
        for d in range(2):
            g[f"out_{lg}_3{d}0"] = g[f"out_{lg}_0{d}0"]
    return g


# ---------------------------------------------------------------- BLS12-381 G2 (oracle/ec2.c)
def fp2_op(op, a, b=None):
    """Element-wise Fp2 op on (n, 12) Montgomery limb arrays: mul, add, sub, sqr, inv."""
    a = np.ascontiguousarray(a, dtype=np.uint64).reshape(-1, 12)
    b = a if b is None else np.ascontiguousarray(b, dtype=np.uint64).reshape(-1, 12)
    r = np.zeros_like(a)
    code = {"mul": 0, "add": 1, "sub": 2, "sqr": 3, "inv": 4}[op]
    for i in range(a.shape[0]):
        lib().oracle_fp2_op(code, _ptr(r[i]), _ptr(a[i]), _ptr(b[i]))
    return r


def g2_points(n):
    """(n, 24) uint64: (i+1)*G2 as affine Montgomery (X.c0, X.c1, Y.c0, Y.c1)."""
    out = np.zeros((n, 24), dtype=np.uint64)
    lib().oracle_g2_points(_ptr(out), n)
    return out


def g2_msm(points, scalars, algo="buckets"):
    """points (n, 24) packed or (n, 25) arkworks G2Affine (flag word last); scalars (n, 4)."""
    points = np.ascontiguousarray(points, dtype=np.uint64)
    scalars = np.ascontiguousarray(scalars, dtype=np.uint64)
    assert points.shape[1] in (24, 25) and scalars.shape == (points.shape[0], 4)
    out = np.zeros(36, dtype=np.uint64)
    lib().oracle_g2_msm(int(algo != "naive"), _ptr(out), _ptr(points), points.strides[0],
                        int(points.shape[1] == 25), points.shape[0], _ptr(scalars))
    return out


def g2_jac_to_affine(jac):
    out = np.zeros(24, dtype=np.uint64)
    lib().oracle_g2_jac_to_affine(_ptr(out), _ptr(np.ascontiguousarray(jac, dtype=np.uint64)))
    return out


def g2_on_curve(xy):
    return bool(lib().oracle_g2_on_curve(_ptr(np.ascontiguousarray(xy, dtype=np.uint64))))


# ---------------------------------------------------------------- reference builds (_ref)
def ref_path(name):
    p = os.path.join(REF_DIR, name)
    return p if os.path.exists(p) else None


_ref_cpu = None


def ref_cpu():
    """The reference's own msm/pippenger.hpp (CPU) -- None if oracle/_ref was not built."""
    global _ref_cpu
    if _ref_cpu is None:
        p = ref_path("libref_msm_cpu.so")
        if p is None:
            return None
        _ref_cpu = C.CDLL(p)
        _ref_cpu.ref_cpu_mult_pippenger.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_int]
        _ref_cpu.ref_cpu_naive.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    return _ref_cpu


def ref_cpu_msm(points, scalars, nthreads=1, naive=False):
    """BLS12-381 G1 through the reference's CPU mult_pippenger; points (n,12) uint64 packed."""
    r = ref_cpu()
    points = np.ascontiguousarray(points, dtype=np.uint64)
    scalars = np.ascontiguousarray(scalars, dtype=np.uint64)
    assert points.shape[1] == 12 and scalars.shape[1] == 4
    out = np.zeros(18, dtype=np.uint64)
    if naive:
        r.ref_cpu_naive(_ptr(out), _ptr(points), points.shape[0], _ptr(scalars))
    else:
        r.ref_cpu_mult_pippenger(_ptr(out), _ptr(points), points.shape[0], _ptr(scalars), nthreads)
    return out

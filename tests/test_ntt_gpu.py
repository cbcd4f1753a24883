"""GPU parity: CUDA NTT through the C-ABI vs the CPU oracle (bit-exact), plus the
reference's own self-consistency protocol (poc/ntt-cuda/tests/ntt.rs:9-79)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

GL_P = 2**64 - 2**32 + 1
BB_P = 0x78000001


def _rand(field, n, seed):
    rng = np.random.default_rng(seed)
    if field == "gl64":
        return rng.integers(0, GL_P, size=n, dtype=np.uint64)
    return rng.integers(0, BB_P, size=n, dtype=np.uint32)


@pytest.mark.parametrize("field", ["gl64", "bb31"])
@pytest.mark.parametrize("lg", list(range(1, 19)) + [20])
def test_ntt_matches_oracle_all_orders(oracle, field, lg):
    from sppark_b200 import ntt
    x = _rand(field, 1 << lg, lg)
    ofn = oracle.ntt_gl64 if field == "gl64" else oracle.ntt_bb31
    for order in (ntt.NN, ntt.NR, ntt.RN, ntt.RR):
        for inverse in (False, True):
            y = x.copy()
            (ntt.iNTT if inverse else ntt.NTT)(0, y, order)
            ref = ofn(x, order, inverse, nthreads=8)
            assert np.array_equal(y, ref), (field, lg, order, inverse)


@pytest.mark.parametrize("field", ["gl64", "bb31"])
@pytest.mark.parametrize("lg", [3, 10, 13, 17])
def test_coset_matches_oracle(oracle, field, lg):
    from sppark_b200 import ntt
    x = _rand(field, 1 << lg, 100 + lg)
    ofn = oracle.ntt_gl64 if field == "gl64" else oracle.ntt_bb31
    for order in (ntt.NN, ntt.NR, ntt.RN, ntt.RR):
        y = x.copy()
        ntt.coset_NTT(0, y, order)
        assert np.array_equal(y, ofn(x, order, False, True, nthreads=8))
        y = x.copy()
        ntt.coset_iNTT(0, y, order)
        assert np.array_equal(y, ofn(x, order, True, True, nthreads=8))


@pytest.mark.parametrize("field,maxlg", [("gl64", 25), ("bb31", 27)])
def test_reference_self_consistency_protocol(field, maxlg):
    """NN == RR; iNTT(NTT(v)) == v for NN, RR and NR->RN  (tests/ntt.rs:19-42, 55-78)."""
    from sppark_b200 import ntt
    for lg in [1, 2, 5, 11, 12, 13, 16, 21, 23, maxlg]:
        v = _rand(field, 1 << lg, 7 * lg)
        nn = v.copy(); ntt.NTT(0, nn, ntt.NN)
        rr = v.copy(); ntt.NTT(0, rr, ntt.RR)
        if lg <= 23:
            # RR output is the bit-reversal of NN output with bit-reversed input; compare via NR
            nr = v.copy(); ntt.NTT(0, nr, ntt.NR)
            idx = np.array([int(format(i, f"0{lg}b")[::-1], 2) for i in range(1 << lg)]) if lg <= 16 else None
            if idx is not None:
                assert np.array_equal(nr[idx], nn)
        ntt.iNTT(0, nn, ntt.NN)
        assert np.array_equal(nn, v), ("NN", lg)
        ntt.iNTT(0, rr, ntt.RR)
        assert np.array_equal(rr, v), ("RR", lg)
        nr = v.copy(); ntt.NTT(0, nr, ntt.NR); ntt.iNTT(0, nr, ntt.RN)
        assert np.array_equal(nr, v), ("NR-RN", lg)


def test_gl64_2pow24_linearity_and_oracle_sample(oracle):
    """Full metric size (2^24): linearity NTT(a+b) = NTT(a)+NTT(b), and direct evaluation of a
    few output coefficients against the definition."""
    from sppark_b200 import ntt
    lg = 24
    n = 1 << lg
    a = _rand("gl64", n, 1)
    b = _rand("gl64", n, 2)
    s = ((a.astype(object) + b.astype(object)) % GL_P).astype(np.uint64) if False else None
    # modular add without object arrays
    s = a + b
    s = np.where(s < a, s + np.uint64(0xFFFFFFFF), s)
    s = np.where(s >= np.uint64(GL_P), s - np.uint64(GL_P), s)
    fa, fb, fs = a.copy(), b.copy(), s.copy()
    for v in (fa, fb, fs):
        ntt.NTT(0, v, ntt.NN)
    t = fa + fb
    t = np.where(t < fa, t + np.uint64(0xFFFFFFFF), t)
    t = np.where(t >= np.uint64(GL_P), t - np.uint64(GL_P), t)
    assert np.array_equal(t, fs)
    full = oracle.ntt_gl64(a, ntt.NN, nthreads=8)
    assert np.array_equal(full, fa)


def test_bad_arguments_return_errors():
    from sppark_b200 import _lib
    l = _lib.lib()
    buf = np.zeros(4, dtype=np.uint64)
    err = l.compute_ntt(0, buf.ctypes.data, 2, 7, 0, 0)
    assert err.code != 0
    if err.message:
        l.drop_error_message(err.message)
    err = l.compute_ntt(99, buf.ctypes.data, 2, 0, 0, 0)
    assert err.code != 0
    if err.message:
        l.drop_error_message(err.message)
    err = l.compute_ntt(0, buf.ctypes.data, 0, 0, 0, 0)     # lg == 0: no-op success
    assert err.code == 0


def test_matches_reference_gpu_golden():
    """Bit-exact against outputs of the reference's own CUDA NTT recorded on a B200
    (tests/golden/ntt_ref_gpu.npz, made by tests/golden/make_golden.py): every order x direction
    x type; Goldilocks lg 1..10 through compute_ntt, BabyBear lg 1..12 through sppark_b200_ntt."""
    import os
    from sppark_b200 import _lib
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "ntt_ref_gpu.npz"))
    l = _lib.lib()
    for field, top in (("gl64", 10), ("bb31", 12)):
        for lg in range(1, top + 1):
            x = g[f"{field}_in_{lg}"]
            for order in range(4):
                for d in range(2):
                    for t in range(2):
                        y = x.copy()
                        if field == "gl64":
                            _lib.check(l.compute_ntt(0, y.ctypes.data, lg, order, d, t))
                        else:
                            _lib.check(l.sppark_b200_ntt(1, 0, y.ctypes.data, lg, order, d, t))
                        assert np.array_equal(y, g[f"{field}_out_{lg}_{order}{d}{t}"]), (field, lg, order, d, t)


@pytest.mark.parametrize("field", ["gl64", "bb31"])
def test_bb_extension_order(oracle, field):
    """BB (bit-reversed in and out) is this library's extension; checked against the oracle."""
    from sppark_b200 import ntt
    ofn = oracle.ntt_gl64 if field == "gl64" else oracle.ntt_bb31
    for lg in (1, 4, 12, 13, 18):
        x = _rand(field, 1 << lg, 900 + lg)
        for inverse in (False, True):
            y = x.copy()
            (ntt.iNTT if inverse else ntt.NTT)(0, y, ntt.BB)
            assert np.array_equal(y, ofn(x, oracle.BB, inverse, nthreads=8))


def test_babybear_2pow27_field_maximum():
    """BASELINE config 5 asks for a 2^28 BabyBear NTT; p - 1 = 15 * 2^27, so 2^27 is the largest
    domain the field (and the reference: MAX_LG_DOMAIN_SIZE 27, ntt/parameters.cuh:14-15) has.
    Full-size checks without the oracle: round trip through NR/RN, linearity, delta -> ones."""
    from sppark_b200 import ntt
    lg = 27
    n = 1 << lg
    a = _rand("bb31", n, 3)
    v = a.copy()
    ntt.NTT(0, v, ntt.NR)
    ntt.iNTT(0, v, ntt.RN)
    assert np.array_equal(v, a)
    d = np.zeros(n, dtype=np.uint32)
    d[0] = 0x0ffffffe                                   # Montgomery one
    ntt.NTT(0, d, ntt.NN)
    assert (d == 0x0ffffffe).all()
    err = None
    from sppark_b200 import _lib
    e = _lib.lib().sppark_b200_ntt(1, 0, a.ctypes.data, 28, 0, 0, 0)     # 2^28 does not exist
    assert e.code != 0
    if e.message:
        _lib.lib().drop_error_message(e.message)


@pytest.mark.parametrize("fid,name", [(2, "bls12_381_fr"), (3, "vesta_fp"), (4, "pallas_fp"), (5, "bn254_fr"),
                                      (6, "bls12_377_fr")])
def test_ntt_256bit_fields_match_oracle(oracle, fid, name):
    """256-bit Montgomery scalar fields (SURVEY section 8a row n3: the reference's "wide" kernels)."""
    import random
    from sppark_b200 import ntt
    rnd = random.Random(fid)
    p = oracle.ff_consts(name)["p"]
    for lg in (1, 2, 3, 7, 11, 12, 14):
        x = np.array([oracle.int_to_limbs(rnd.randrange(p), 4) for _ in range(1 << lg)], dtype=np.uint64)
        for order in (ntt.NN, ntt.NR, ntt.RN, ntt.RR, ntt.BB):
            for inverse in (False, True):
                y = x.copy()
                (ntt.iNTT if inverse else ntt.NTT)(0, y, order, field=fid)
                assert np.array_equal(y, oracle.ntt_ff(name, x, order, inverse)), (name, lg, order, inverse)
        if lg in (3, 12):
            for order in (ntt.NN, ntt.NR, ntt.RN, ntt.RR):
                y = x.copy(); ntt.coset_NTT(0, y, order, field=fid)
                assert np.array_equal(y, oracle.ntt_ff(name, x, order, False, True))
                y = x.copy(); ntt.coset_iNTT(0, y, order, field=fid)
                assert np.array_equal(y, oracle.ntt_ff(name, x, order, True, True))


def test_ntt_256bit_matches_reference_gpu_golden():
    """BLS12-381 scalar field, lg 1..10, every order x direction x type, against the recording of
    the reference's own 256-bit ("wide") CUDA kernels."""
    import os
    from sppark_b200 import ntt
    from oracle import pyoracle
    g = pyoracle.ntt256_golden(os.path.join(os.path.dirname(__file__), "golden", "ntt256_ref_gpu.npz"))
    for lg in range(1, 11):
        x = g[f"in_{lg}"]
        for order in range(4):
            for d in range(2):
                for t in range(2):
                    y = x.copy()
                    ntt._run(0, y, order, d, t, field=ntt.BLS12_381_FR)
                    assert np.array_equal(y, g[f"out_{lg}_{order}{d}{t}"]), (lg, order, d, t)


def test_ntt_256bit_2pow22_roundtrip():
    import random
    from sppark_b200 import ntt
    lg = 22
    rng = np.random.default_rng(9)
    x = rng.integers(0, 2**62, size=(1 << lg, 4), dtype=np.uint64)      # < 2^254: valid residues
    y = x.copy()
    ntt.NTT(0, y, ntt.NR, field=ntt.BLS12_381_FR)
    ntt.iNTT(0, y, ntt.RN, field=ntt.BLS12_381_FR)
    assert np.array_equal(x, y)


@pytest.mark.parametrize("field,lg,lg_g", [("gl64", 16, 1), ("gl64", 20, 3), ("bb31", 18, 2), ("gl64", 24, 3),
                                           ("gl64", 25, 1), ("bb31", 26, 2), ("bb31", 27, 3)])
def test_slab_sharded_transform_on_one_gpu(oracle, field, lg, lg_g):
    """The multi-GPU NTT with its G ranks run one after another on this GPU (the exchange is a
    tensor shuffle): both CUDA stages + layouts against the oracle's single-array transform.
    Above 2^24 the second stage is two passes (BabyBear 2^27, the field's maximum, is SURVEY.md
    section 8d config 5: 2^9 x 2^18 over 8 ranks)."""
    import torch
    from sppark_b200 import ntt, parallel
    G = 1 << lg_g
    fid = 0 if field == "gl64" else 1
    x = _rand(field, 1 << lg, lg + lg_g)
    tdt = torch.int64 if field == "gl64" else torch.int32
    sdt = np.int64 if field == "gl64" else np.int32
    staged = []
    for r in range(G):
        loc = torch.from_numpy(parallel.scatter_columns(x, lg, lg_g, r, fid).reshape(-1).view(sdt).copy()).cuda()
        st = torch.empty_like(loc)
        parallel.gpu_slab_pass(fid, lg, lg_g, r)(1, loc, st)
        staged.append(st.view(G, -1))
    outs = []
    for r in range(G):
        recv = torch.cat([staged[q][r] for q in range(G)]).contiguous()
        parallel.gpu_slab_pass(fid, lg, lg_g, r)(2, recv, torch.empty_like(recv) if lg > 24 else recv)
        outs.append(recv.cpu().numpy().view(x.dtype))
    got = parallel.gather_columns(outs, lg, lg_g, fid)
    ofn = oracle.ntt_gl64 if field == "gl64" else oracle.ntt_bb31
    assert np.array_equal(got, ofn(x, oracle.NN, nthreads=16))


@pytest.mark.parametrize("field,lg,lg_g", [("gl64", 16, 1), ("gl64", 20, 3), ("bb31", 18, 2), ("gl64", 24, 3), ("bb31", 25, 3)])
def test_slab_fused_exchange_on_one_gpu(oracle, field, lg, lg_g):
    """sppark_b200_ntt_slab_pass_p2p: stage 1 stores its rows straight into the receivers' buffers
    (NVLink peer memory between processes; here the G receivers are G allocations of this GPU,
    one of them through the library's peer_alloc).  No staging buffer, no exchange step."""
    import ctypes as C
    import torch
    from sppark_b200 import _lib, parallel
    G = 1 << lg_g
    fid = 0 if field == "gl64" else 1
    x = _rand(field, 1 << lg, lg + lg_g + 1)
    tdt = torch.int64 if field == "gl64" else torch.int32
    sdt = np.int64 if field == "gl64" else np.int32
    n_local = (1 << lg) // G
    peers = parallel.SlabPeers(n_local * x.dtype.itemsize, nbuf=1)          # world = 1: owns one buffer
    recv = [peers.tensor(0, tdt)] + [torch.empty(n_local, dtype=tdt, device="cuda") for _ in range(G - 1)]
    ptrs = (C.c_void_p * G)(*[t.data_ptr() for t in recv])
    stream = torch.cuda.current_stream().cuda_stream
    for r in range(G):
        loc = torch.from_numpy(parallel.scatter_columns(x, lg, lg_g, r, fid).reshape(-1).view(sdt).copy()).cuda()
        _lib.check(_lib.lib().sppark_b200_ntt_slab_pass_p2p(fid, loc.data_ptr(), ptrs, lg, lg_g, r, 0, stream))
    outs = []
    scratch = torch.empty(n_local, dtype=tdt, device="cuda")
    for r in range(G):
        parallel.gpu_slab_pass(fid, lg, lg_g, r)(2, recv[r], scratch)
        outs.append(recv[r].cpu().numpy().view(x.dtype))
    got = parallel.gather_columns(outs, lg, lg_g, fid)
    peers.close()
    ofn = oracle.ntt_gl64 if field == "gl64" else oracle.ntt_bb31
    assert np.array_equal(got, ofn(x, oracle.NN, nthreads=16))


def test_gpu_ptr_handles():
    """clone_gpu_ptr_t / drop_gpu_ptr_t keep the reference's ownership protocol
    (util/gpu_t.cuh:268-316): the memory lives until the last handle is dropped."""
    import ctypes as C
    import torch
    from sppark_b200 import _lib, ntt
    l = _lib.lib()
    h = l.sppark_b200_gpu_ptr_alloc(1 << 20)
    assert h.inner and l.sppark_b200_gpu_ptr_refs(C.byref(h)) == 1
    h2 = l.clone_gpu_ptr_t(C.byref(h))
    assert h2.inner == h.inner and l.sppark_b200_gpu_ptr_refs(C.byref(h)) == 2
    dptr = l.sppark_b200_gpu_ptr_get(C.byref(h2))
    l.drop_gpu_ptr_t(C.byref(h))
    assert not h.inner and l.sppark_b200_gpu_ptr_refs(C.byref(h2)) == 1
    # the allocation is still usable through the surviving handle: run an NTT in it
    x = _rand("gl64", 1 << 10, 1)
    t = torch.from_numpy(x.view(np.int64)).cuda()
    _lib.check(l.sppark_b200_ntt_dev(0, dptr, 10, 0, 0, 0, None)) if False else None
    l.drop_gpu_ptr_t(C.byref(h2))
    assert not h2.inner


@pytest.mark.parametrize("field,fid", [("gl64", 0), ("bb31", 1), ("bls12_381_fr", 2)])
def test_lde_matches_definition(oracle, field, fid):
    """NTT::LDE / LDE_aux (SURVEY section 8f row 1): extended coset evaluations + coefficients."""
    import random
    from sppark_b200 import ntt
    rnd = random.Random(fid)
    for lg, lb in ((1, 1), (5, 1), (8, 3), (12, 2), (13, 1), (16, 2)):
        if field in ("gl64", "bb31"):
            x = _rand(field, 1 << lg, lg * 7 + lb)
        else:
            p = oracle.ff_consts(field)["p"]
            if lg > 12:
                continue
            x = np.array([oracle.int_to_limbs(rnd.randrange(p), 4) for _ in range(1 << lg)], dtype=np.uint64)
        ext, coeffs = ntt.LDE(0, x, lb, field=fid, want_coefficients=True)
        want_ext, want_c = oracle.lde(field, x, lb)
        assert np.array_equal(coeffs, want_c), (field, lg, lb)
        assert np.array_equal(ext, want_ext), (field, lg, lb)


def test_lde_matches_reference_gpu_golden():
    import os
    from sppark_b200 import ntt
    path = os.path.join(os.path.dirname(__file__), "golden", "lde_ref_gpu.npz")
    if not os.path.exists(path):
        pytest.skip("golden not recorded yet")
    g = np.load(path)
    for lg, lb in ((1, 1), (3, 1), (6, 2), (10, 1), (12, 3)):
        assert np.array_equal(ntt.LDE(0, g[f"in_{lg}_{lb}"], lb), g[f"out_{lg}_{lb}"]), (lg, lb)


def _word_selftest(field, op, a, b):
    from sppark_b200 import _lib
    a = np.ascontiguousarray(a)
    b = np.ascontiguousarray(b)
    r = np.zeros_like(a)
    _lib.check(_lib.lib().sppark_b200_selftest_word_field(field, op, a.size, r.ctypes.data, a.ctypes.data, b.ctypes.data))
    return r


def _gl64_operands(seed, n):
    """Pairs (a loose, b canonical) with every carry / borrow / wrap corner of p = 2^64 - 2^32 + 1."""
    edge = [0, 1, 2, 0xFFFFFFFE, 0xFFFFFFFF, 0x100000000, 0x100000001, 2**63 - 1, 2**63, 2**63 + 1,
            0xFFFFFFFE00000000, 0xFFFFFFFEFFFFFFFF, 0xFFFFFFFF00000000, GL_P - 1, GL_P, GL_P + 1,
            0xFFFFFFFF00000002, 0xFFFFFFFFFFFFFFFE, 0xFFFFFFFFFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF00000001 - 0xFFFFFFFF]
    a = [x for x in edge for _ in edge]
    b = [y % GL_P for _ in edge for y in edge]
    rng = np.random.default_rng(seed)
    ra = rng.integers(0, 2**64, size=n, dtype=np.uint64)
    rb = rng.integers(0, GL_P, size=n, dtype=np.uint64)
    # operands with saturated halves hit the +-EPS corrections far more often than uniform ones
    ra[: n // 4] |= np.uint64(0xFFFFFFFF00000000)
    rb[n // 8: n // 4] = (rb[n // 8: n // 4] | np.uint64(0xFFFFFFFE00000000)) % np.uint64(GL_P)
    return (np.concatenate([np.array(a, dtype=np.uint64), ra]), np.concatenate([np.array(b, dtype=np.uint64), rb]))


def test_gl64_device_field_arithmetic_known_answers():
    """The PTX field arithmetic against Python integers: add / sub keep the value mod p for a loose
    first and a canonical second operand; mul is the Montgomery product a*b*2^-64 and is canonical;
    tight / canon reduce below p."""
    a, b = _gl64_operands(11, 1 << 16)
    ai = [int(v) for v in a]
    bi = [int(v) for v in b]
    rinv = pow(2**64, -1, GL_P)
    got = _word_selftest(0, 1, a, b)
    assert all(int(g) % GL_P == (x + y) % GL_P for g, x, y in zip(got, ai, bi))
    got = _word_selftest(0, 2, a, b)
    assert all(int(g) % GL_P == (x - y) % GL_P for g, x, y in zip(got, ai, bi))
    got = _word_selftest(0, 0, a, b)
    assert all(int(g) == x * y * rinv % GL_P for g, x, y in zip(got, ai, bi))
    for op in (3, 4):
        got = _word_selftest(0, op, a, b)
        assert all(int(g) == x % GL_P for g, x in zip(got, ai))


def test_bb31_device_field_arithmetic_known_answers():
    rng = np.random.default_rng(12)
    edge = np.array([0, 1, 2, BB_P - 1, BB_P - 2, BB_P // 2, BB_P // 2 + 1, 0x0FFFFFFE], dtype=np.uint32)
    a = np.concatenate([np.repeat(edge, len(edge)), rng.integers(0, BB_P, size=1 << 14, dtype=np.uint32)])
    b = np.concatenate([np.tile(edge, len(edge)), rng.integers(0, BB_P, size=1 << 14, dtype=np.uint32)])
    ai = a.astype(np.uint64)
    bi = b.astype(np.uint64)
    assert np.array_equal(_word_selftest(1, 1, a, b), ((ai + bi) % BB_P).astype(np.uint32))
    assert np.array_equal(_word_selftest(1, 2, a, b), ((ai + BB_P - bi) % BB_P).astype(np.uint32))
    rinv = pow(2**32, -1, BB_P)
    want = np.array([int(x) * int(y) * rinv % BB_P for x, y in zip(a, b)], dtype=np.uint32)
    assert np.array_equal(_word_selftest(1, 0, a, b), want)


@pytest.mark.parametrize("field", ["gl64", "bb31"])
@pytest.mark.parametrize("split", ["4,4,4", "5,5,5", "6,6", "7,7,7", "8,8", "8,4,6", "4,5,4,5"])
def test_warp_pass_every_subntt_size(oracle, field, split, monkeypatch):
    """Every sub-NTT size of the warp-autonomous pass (2^4..2^8), in every position of a plan and
    in every order / direction, against the oracle."""
    from sppark_b200 import ntt
    monkeypatch.setenv("SPPARK_B200_NTT_SPLIT", split)
    monkeypatch.setenv("SPPARK_B200_NTT_WARP", "1")
    lg = sum(int(v) for v in split.split(","))
    x = _rand(field, 1 << lg, 900 + lg)
    ofn = oracle.ntt_gl64 if field == "gl64" else oracle.ntt_bb31
    for order in (ntt.NN, ntt.NR, ntt.RN, ntt.RR):
        for inverse in (False, True):
            y = x.copy()
            (ntt.iNTT if inverse else ntt.NTT)(0, y, order)
            assert np.array_equal(y, ofn(x, order, inverse, nthreads=8)), (field, split, order, inverse)


@pytest.mark.parametrize("cpt", ["1", "2"])
@pytest.mark.parametrize("field", ["gl64", "bb31"])
def test_warp_pass_columns_per_lane(oracle, field, cpt, monkeypatch):
    from sppark_b200 import ntt
    monkeypatch.setenv("SPPARK_B200_NTT_CPT", cpt)
    monkeypatch.setenv("SPPARK_B200_NTT_WARP", "1")
    ofn = oracle.ntt_gl64 if field == "gl64" else oracle.ntt_bb31
    for lg in (4, 5, 9, 13, 16, 19):
        x = _rand(field, 1 << lg, 70 + lg)
        for order in (ntt.NN, ntt.NR, ntt.RN):
            for inverse in (False, True):
                y = x.copy()
                (ntt.iNTT if inverse else ntt.NTT)(0, y, order)
                assert np.array_equal(y, ofn(x, order, inverse, nthreads=8)), (field, cpt, lg, order, inverse)


@pytest.mark.parametrize("field", ["gl64", "bb31"])
@pytest.mark.parametrize("knob,sizes", [("SPPARK_B200_NTT_BLOCK", [4, 9, 13, 17]), ("SPPARK_B200_NTT_WARP", [20, 22])])
def test_both_pass_kernels_at_every_size_class(oracle, field, knob, sizes, monkeypatch):
    """The library picks the warp-autonomous passes below 2^20 and the block-tile passes above;
    each kernel is also correct on the other side of that line."""
    from sppark_b200 import ntt
    monkeypatch.setenv(knob, "1")
    ofn = oracle.ntt_gl64 if field == "gl64" else oracle.ntt_bb31
    for lg in sizes:
        x = _rand(field, 1 << lg, 300 + lg)
        for order in (ntt.NN, ntt.NR, ntt.RN):
            for inverse in (False, True):
                y = x.copy()
                (ntt.iNTT if inverse else ntt.NTT)(0, y, order)
                assert np.array_equal(y, ofn(x, order, inverse, nthreads=8)), (field, knob, lg, order, inverse)


@pytest.mark.parametrize("field", ["gl64", "bb31"])
@pytest.mark.parametrize("chunks", [1, 2, 4, 8])
def test_ntt_sharded_c_abi_on_one_device(oracle, field, chunks):
    """sppark_b200_ntt_sharded (single process, C ABI): every chunk on device 0, so the exchange
    runs as block copies; bit-exact against the oracle, forward and inverse, including sizes whose
    second stage takes several passes."""
    from sppark_b200 import parallel
    ofn = oracle.ntt_gl64 if field == "gl64" else oracle.ntt_bb31
    for lg in (6, 13, 20) + ((25,) if chunks == 8 and field == "bb31" else ()):
        x = _rand(field, 1 << lg, 40 + lg)
        y = x.copy()
        parallel.ntt_sharded_c(y, [0] * chunks)
        assert np.array_equal(y, ofn(x, 0, False, nthreads=8)), (field, chunks, lg)
        parallel.ntt_sharded_c(y, [0] * chunks, inverse=True)
        assert np.array_equal(y, x), (field, chunks, lg, "inverse")


def test_ntt_sharded_c_abi_across_devices(oracle):
    """Fused exchange (NVLink peer stores) when this box has at least two GPUs that see each other."""
    import torch
    from sppark_b200 import parallel
    ndev = torch.cuda.device_count()
    if ndev < 2:
        pytest.skip("one GPU")
    g = 1 << (min(ndev, 8).bit_length() - 1)
    for field, ofn in (("gl64", oracle.ntt_gl64), ("bb31", oracle.ntt_bb31)):
        for lg in (13, 22):
            x = _rand(field, 1 << lg, 60 + lg)
            y = x.copy()
            parallel.ntt_sharded_c(y, list(range(g)))
            assert np.array_equal(y, ofn(x, 0, False, nthreads=8)), (field, lg)
            parallel.ntt_sharded_c(y, list(range(g)), inverse=True)
            assert np.array_equal(y, x)


@pytest.mark.parametrize("field", ["gl64", "bb31"])
def test_lde_device_entries_compose_to_the_host_lde(oracle, field):
    """NTT::LDE_powers / LDE_expand on device memory (ntt/ntt.cuh:352-365): iNTT(NR), powers,
    expand (in place: the coefficients sit at the tail of the extended buffer), NTT(RN) must equal
    the one-call LDE, which is pinned against the reference's own recording."""
    import torch
    from sppark_b200 import _lib, ntt
    l = _lib.lib()
    fid, tdt = (0, torch.int64) if field == "gl64" else (1, torch.int32)
    for lg, lb in ((5, 1), (10, 2), (14, 3)):
        n, n_ext = 1 << lg, 1 << (lg + lb)
        x = _rand(field, n, 500 + lg)
        want, coeffs = ntt.LDE(0, x, lb, want_coefficients=True)
        ext = torch.zeros(n_ext, dtype=tdt, device="cuda")
        tail = ext[n_ext - n:]
        tail.copy_(torch.from_numpy(x.view(np.int64 if field == "gl64" else np.int32)))
        s = torch.cuda.current_stream().cuda_stream
        _lib.check(l.sppark_b200_ntt_dev(fid, tail.data_ptr(), lg, ntt.NR, ntt.INVERSE, 0, s))
        _lib.check(l.sppark_b200_lde_powers_dev(fid, tail.data_ptr(), lg, s))
        _lib.check(l.sppark_b200_lde_expand_dev(fid, ext.data_ptr(), tail.data_ptr(), lg, lb, s))
        _lib.check(l.sppark_b200_ntt_dev(fid, ext.data_ptr(), lg + lb, ntt.RN, ntt.FORWARD, 0, s))
        torch.cuda.synchronize()
        got = ext.cpu().numpy().view(x.dtype)
        assert np.array_equal(got, want), (field, lg, lb)
        # the natural-order coefficients of LDE_aux: inverse transform of the evaluations
        y = x.copy()
        ntt.iNTT(0, y, ntt.NN)
        assert np.array_equal(coeffs, y), (field, lg, lb)

"""CPU builds (g++) of the product's field / curve headers against the oracle, without a GPU, in two variants:
"portable" = the plain C++ arithmetic path; "emulated" = the device's carry-chain formulation (the source ptxas sees,
-DGMSM_EMULATE_PTX: mad.lo.cc / madc.hi.cc / addc ... over an emulated carry flag, dropped carries trap).  The PTX itself
is checked by the same vectors on the GPU in tests/test_gpu_ops.py and tests/test_gpu_arith_edges.py."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle import oracle as O
from tests import opcases

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "gnark-crypto_b200", "csrc")
OUT = os.path.join(ROOT, "gnark-crypto_b200", "build", "libgmsm_hostcheck%s.so")
_LIBS = {}


def _build(variant):
    """per-group objects + the dispatcher, compiled in parallel; rebuilt only when a header is newer than the .so"""
    if variant not in _LIBS:
        tag = {"portable": "", "emulated": "_emu", "emulated_sqr": "_emusqr", "emulated_fp2dot": "_emufp2dot", "emulated_fp2lazy": "_emufp2lazy", "portable_fp2lazy": "_fp2lazy", "emulated_kara": "_emukara", "portable_kara": "_kara", "emulated_dot4": "_emudot4"}[variant]
        out = OUT % tag
        bdir = os.path.dirname(out)
        os.makedirs(bdir, exist_ok=True)
        srcs = [os.path.join(CSRC, n) for n in os.listdir(CSRC) if n.endswith((".cuh", ".h", ".cpp"))]
        if not os.path.exists(out) or os.path.getmtime(out) < max(os.path.getmtime(p) for p in srcs):
            flags = ["-std=c++17", "-O1", "-fPIC"] + {"portable": [], "emulated": ["-DGMSM_EMULATE_PTX"],
                                                     "emulated_sqr": ["-DGMSM_EMULATE_PTX", "-DGMSM_SQR_DEDICATED=1", "-DGMSM_DOT2=1"],
                                                     "emulated_fp2dot": ["-DGMSM_EMULATE_PTX", "-DGMSM_SQR_DEDICATED=1", "-DGMSM_DOT2=1", "-DGMSM_FP2_DOT2=1"],
                                                     "emulated_fp2lazy": ["-DGMSM_EMULATE_PTX", "-DGMSM_FP2_LAZY=1"], "portable_fp2lazy": ["-DGMSM_FP2_LAZY=1"],
                                                     "emulated_kara": ["-DGMSM_EMULATE_PTX", "-DGMSM_MUL_KARATSUBA=1", "-DGMSM_SQR_DEDICATED=1", "-DGMSM_DOT2=1"],
                                                     "portable_kara": ["-DGMSM_MUL_KARATSUBA=1"],
                                                     "emulated_dot4": ["-DGMSM_EMULATE_PTX", "-DGMSM_SQR_DEDICATED=1", "-DGMSM_DOT2=1", "-DGMSM_FP2_DOT2=1", "-DGMSM_DOT4=1"]}[variant]
            src = os.path.join(CSRC, "hostcheck.cpp")
            objs, procs = [], []
            for k in list(range(len(O.GROUPS) + 1)) + [None]:     # + the field-only pseudo group (secp256k1 fr)
                o = os.path.join(bdir, "hostcheck%s_%s.o" % (tag, "d" if k is None else k))
                objs.append(o)
                procs.append(subprocess.Popen(["g++", *flags, *([] if k is None else ["-DHC_GROUP=%d" % k]), "-c", "-o", o, src]))
            assert all(p.wait() == 0 for p in procs)
            subprocess.run(["g++", "-shared", "-o", out, *objs], check=True)
        _LIBS[variant] = ctypes.CDLL(out)
    return _LIBS[variant]


# "emulated_sqr": the experimental dedicated squaring and fused two-product routine of field.cuh
# (-DGMSM_SQR_DEDICATED=1 -DGMSM_DOT2=1, not in the default build); the point formulas of curve.cuh then use them
# "emulated_kara" / "portable_kara": the field product as REDC(one-level Karatsuba) (-DGMSM_MUL_KARATSUBA=1)
# "emulated_fp2lazy" / "portable_fp2lazy": the Fp2 product with lazy reduction over the separated wide product / REDC routines (-DGMSM_FP2_LAZY=1)
# "emulated_dot4": additionally the four-product fused reduction behind the Fp2 y-coordinate (-DGMSM_DOT4=1, shipped for bn254 G2)
# "emulated_fp2dot": additionally the Fp2 product as two fused two-product reductions (fp2.cuh, -DGMSM_FP2_DOT2=1)
# The variants of routines that are NOT in the shipped build (lazy-reduction Fp2 product, Karatsuba product: measured slower,
# DESIGN.md section 2) run only with GMSM_TEST_EXPERIMENTAL=1, to keep the CPU suite within a few minutes.
_VARIANTS = ["portable", "emulated", "emulated_sqr", "emulated_fp2dot", "emulated_dot4"] + (
    ["emulated_fp2lazy", "portable_fp2lazy", "emulated_kara", "portable_kara"] if os.environ.get("GMSM_TEST_EXPERIMENTAL") else [])


@pytest.fixture(scope="module", params=_VARIANTS)
def hc(request):
    return _build(request.param)


def _runner(hc, g):
    cid = len(O.GROUPS) if g == "secp256k1_fr" else list(O.GROUPS).index(g)
    assert list(O.GROUPS) == ["bn254_g1", "bn254_g2", "bls12381_g1", "bls12381_g2", "bls12377_g1", "bls12377_g2", "secp256k1_g1",
                              "bw6761_g1", "bw6761_g2", "bls24315_g1", "bls24317_g1", "bw6633_g1", "bw6633_g2"]

    def run(op, a, b, out_words):
        a = np.ascontiguousarray(a, dtype=np.uint32)
        n = a.shape[0]
        b = np.ascontiguousarray(b, dtype=np.uint32) if b is not None else np.zeros((n, 1), dtype=np.uint32)
        out = np.zeros((n, out_words), dtype=np.uint32)
        rc = hc.hostcheck_op(cid, op, a.ctypes.data_as(ctypes.c_void_p), b.ctypes.data_as(ctypes.c_void_p),
                             out.ctypes.data_as(ctypes.c_void_p), ctypes.c_size_t(n))
        assert rc == 0
        return out

    return run


@pytest.mark.parametrize("g", list(O.GROUPS))
def test_field_ops_host(hc, g):
    opcases.check_field_ops(O.GROUPS[g], _runner(hc, g))
    opcases.check_fr_from_mont(O.GROUPS[g], _runner(hc, g))


@pytest.mark.parametrize("g", list(O.GROUPS))
def test_field_edges_host(hc, g):
    """extreme operands (opcases.extreme_values) through every coordinate-field op, the fused sums of two and four products
    and the inversion, against big-integer arithmetic on the raw limbs: each variant's formulation of the carry chains"""
    opcases.check_field_edges(O.GROUPS[g], _runner(hc, g), n_random=64, n_perm=3)


@pytest.mark.parametrize("g", list(O.GROUPS))
def test_point_ops_host(hc, g):
    opcases.check_point_ops(O.GROUPS[g], _runner(hc, g))
    opcases.check_point_edges(O.GROUPS[g], _runner(hc, g))


@pytest.mark.parametrize("g,c", [("bn254_g1", 5), ("bn254_g1", 22), ("bn254_g2", 7), ("bls12381_g1", 11), ("bls12381_g2", 3),
                                 ("bls12377_g1", 9), ("bls12377_g2", 4), ("secp256k1_g1", 8), ("bw6761_g1", 6), ("bw6761_g2", 5),
                                 ("bls24315_g1", 7), ("bls24317_g1", 10), ("bw6633_g1", 6), ("bw6633_g2", 9)])
def test_table_level_host(hc, g, c):
    """one level of the window tables (k_table_level's batch function, built for the CPU): out_i = 2^c * in_i in affine
    normal form, infinity preserved, ragged batch (19 = 2 full batches of 8 + 3)"""
    G = O.GROUPS[g]
    pts = O.consecutive_multiples(G, 19, start_k=3)
    pts[4] = G.aff_inf()
    pts[16] = G.aff_inf()
    pts[9] = pts[8]
    arr = np.ascontiguousarray(G.encode_affine(pts)).view(np.uint32).reshape(19, -1)
    out = np.zeros_like(arr)
    rc = hc.hostcheck_table_level(list(O.GROUPS).index(g), c, arr.ctypes.data_as(ctypes.c_void_p), ctypes.c_size_t(19),
                                  out.ctypes.data_as(ctypes.c_void_p))
    assert rc == 0
    want = [G.aff_inf() if G.aff_is_inf(p) else G.scalar_mul(p, 1 << c) for p in pts]
    assert np.array_equal(out.view(np.uint64).reshape(19, -1), G.encode_affine(want))
    # all-infinity batch: the shared inversion runs on the empty product
    z = np.zeros_like(arr[:5])
    o2 = np.ones_like(z)
    assert hc.hostcheck_table_level(list(O.GROUPS).index(g), c, z.ctypes.data_as(ctypes.c_void_p), ctypes.c_size_t(5),
                                    o2.ctypes.data_as(ctypes.c_void_p)) == 0
    assert not o2.any()


def test_window_plan(hc):
    buf = (ctypes.c_int * 6)()
    for bits in (253, 254, 255, 256, 315, 377):
        for c in range(2, 25):
            hc.hostcheck_plan(bits, c, buf)
            W = O.compute_nb_chunks(bits, c)
            lc = O.last_c(bits, c)
            assert list(buf) == [c, W, lc, 1 << (c - 1), 1 << (lc - 1), (W - 1) * (1 << (c - 1)) + (1 << (lc - 1))]


@pytest.mark.parametrize("g", ["bn254_g1", "bls12381_g1", "bls12377_g1", "secp256k1_g1", "secp256k1_fr", "bw6761_g1", "bls24315_g1",
                               "bls24317_g1", "bw6633_g1"])
def test_carry_chain_mul_sqr_stress(g):
    """the device formulation of Mul / Square (emulated) against the portable path and big-int arithmetic on many random
    and extreme operands (limbs of all-ones, single bits, q-1, values next to the limb boundaries).  secp256k1's two moduli
    fill all 256 bits: the multiplier keeps the carries a spare top bit would make zero (field.cuh, P::FULL)"""
    f = O.FIELDS[g] if g.endswith("_fr") else O.GROUPS[g].K.f
    rng = np.random.default_rng(17)
    nl = f.limbs * 2
    import random
    r = random.Random(5)
    vals = opcases.extreme_values(f) + [r.randrange(f.q) for _ in range(3000)]
    A = np.array([f.to_limbs(v) for v in vals], dtype=np.uint64).view(np.uint32).reshape(len(vals), nl)
    perm = rng.permutation(len(vals))
    B = A[perm]
    run_p, run_e = _runner(_build("portable"), g), _runner(_build("emulated"), g)
    mp, me = run_p(0, A, B, nl), run_e(0, A, B, nl)
    sp, se = run_p(3, A, None, nl), run_e(3, A, None, nl)
    assert np.array_equal(mp, me) and np.array_equal(sp, se)
    # the experimental dedicated squaring (rows restricted to the limbs j >= i, doubled operand above the diagonal)
    sq = _runner(_build("emulated_sqr"), g)(3, A, None, nl)
    assert np.array_equal(sq, sp)
    # the experimental fused two-product routine: (x*y + u*v) R^-1 with one reduction, against big-int arithmetic and
    # against its plain composition (two products and an addition) in the portable build
    C, D = A[rng.permutation(len(vals))], A[rng.permutation(len(vals))]
    cid = len(O.GROUPS) if g == "secp256k1_fr" else list(O.GROUPS).index(g)
    outs = []
    for variant in ("portable", "emulated_sqr"):
        out = np.zeros_like(A)
        vp = ctypes.c_void_p
        assert _build(variant).hostcheck_dot2(cid, A.ctypes.data_as(vp), B.ctypes.data_as(vp), C.ctypes.data_as(vp), D.ctypes.data_as(vp),
                                              out.ctypes.data_as(vp), ctypes.c_size_t(len(vals))) == 0
        outs.append(out)
    assert np.array_equal(outs[0], outs[1])
    lim = lambda M: [f.from_limbs(row) for row in np.ascontiguousarray(M).view(np.uint64)]
    a_, b_, c_, d_ = lim(A), lim(B), lim(C), lim(D)
    assert lim(outs[1]) == [(x * y + u * v) * f.Rinv % f.q for x, y, u, v in zip(a_, b_, c_, d_)]
    # additions / doublings / subtractions of the same extreme operands (full-width moduli: the carry out of the limbs decides
    # the final subtraction, field.cuh fp_reduce_once)
    for op, fn in ((1, lambda x, y: (x + y) % f.q), (2, lambda x, y: (x - y) % f.q)):
        for run in (run_p, run_e):
            assert lim(run(op, A, B, nl)) == [fn(x, y) for x, y in zip(a_, b_)]
    assert lim(run_e(5, A, None, nl)) == [2 * x % f.q for x in a_]
    # inversion (binary GCD; for the full-width moduli the bit of y + q above the limbs is shifted back in): inv(xR) = x^-1 R
    sel = list(range(0, len(vals), 17))
    inv = lim(run_e(6, A[sel], None, nl))
    assert inv == [(pow(a_[i], -1, f.q) * f.R2 % f.q) if a_[i] else 0 for i in sel]
    got_m = [f.from_limbs(row) for row in me.view(np.uint64)]
    got_s = [f.from_limbs(row) for row in se.view(np.uint64)]
    assert got_m == [vals[i] * vals[perm[i]] * f.Rinv % f.q for i in range(len(vals))]
    assert got_s == [v * v * f.Rinv % f.q for v in vals]

"""MultiExp past 2^31 bucket entries, up to the largest n * W a context accepts.

The bucket pipeline numbers its entries (one per non-zero digit) with 32-bit indices: a context accepts n with
n * W < 4,294,967,000, which with chunks of K <= 256 entries also keeps the end of the last accumulate chunk, start + K, below
2^32.  Past 2^31 entries a signed 32-bit index, a u32 product or an unwidened sum goes wrong silently, so each case here runs one
device-level MultiExp with more than 2^31 entries (counted from the digits of its scalars, not just n * W) -- K1 (plain and rank
mode), the scan, the per-window scatter (the split part on the auxiliary stream), both k_accumulate launches, the carry levels,
bucket reduction and finalize -- and compares the point limb for limb with the oracle.

Inputs without multi-GB host arrays: bases [i+1]B generated on the device, scalars s_i = S[i mod P] tiled on the device from a
table of P random scalars.  The expected scalar is then exact in Python over the P table entries:
    k = sum_j fromMont(S_j) * sum_{i < n, i = j mod P} (i + 1)  (mod r),   the inner sum = m(j+1) + P m(m-1)/2, m = ceil((n-j)/P)
and the expected point [k]B comes from the oracle's C port; nothing in it uses the engine's field code.

Each case needs 44..66 GB of device memory by the estimate below.  It is skipped, with both numbers in the reason, only when the
device does not have that much free before the case starts; an engine error with the memory there is a failure."""
import importlib

import numpy as np
import pytest

from oracle import cref
from oracle import oracle as O

pytestmark = pytest.mark.gpu

ENTRY_LIMIT = 4_294_967_000         # n * W of one context (ctx_create_ex, gmsm.cu)
TABLE_LIMIT = 2_147_483_000         # row_stride * W of a window table
P = 1_000_003                       # period of the scalar table (prime, so that i mod P mixes every window's digits)
HI_SLOT = (1 << 31) + 12345         # a slot past 2^31 of the chunk-major digit / rank arrays (digits[j*n + i])


def _pkg():
    import gnark_crypto_b200 as pkg

    return pkg


def _mx():
    return importlib.import_module("gnark-crypto_b200.multiexp")


def _native():
    return importlib.import_module("gnark-crypto_b200._native")


def _nwin(g, c):
    bits = _mx().SCALAR_BITS[_mx().CURVES[g]]
    return (bits + c - 1) // c


def _estimate_bytes(g, n, c):
    """device memory of one case: digits, ranks and entries (12 bytes per entry), points, scalars, the two carry levels and the
    buckets of the context, plus 10 %"""
    cid = _mx().CURVES[g]
    L = _native().lib()
    bits = _mx().SCALAR_BITS[cid]
    W = _nwin(g, c)
    last_c = c + 1 - (W * c - bits)
    nb_total = (W - 1) * (1 << (c - 1)) + (1 << (last_c - 1))
    ent = n * W
    chunks = max(700_000, ent // 128 + 1)           # chunks of the accumulate kernel (ctx_alloc), K2_first = 4 for level two
    xyzz = L.gmsm_xyzz_bytes(cid)
    need = 12 * ent + n * (L.gmsm_affine_bytes(cid) + L.gmsm_scalar_bytes(cid)) + (chunks + chunks // 4) * (xyzz + 4) + nb_total * xyzz
    return int(need * 1.1)


def _require_memory(g, n, c):
    import torch

    torch.cuda.empty_cache()
    need = _estimate_bytes(g, n, c)
    free, _ = torch.cuda.mem_get_info()
    if free < need:
        pytest.skip("needs ~%.1f GB of device memory, %.1f GB free" % (need / 1e9, free / 1e9))


def _expected_scalar(G, table, n):
    """sum_i (i + 1) * S[i mod P] mod r over i < n, exact"""
    s = G.decode_scalars(table)
    p = len(s)
    k = 0
    for j in range(min(p, n)):
        m = (n - j + p - 1) // p
        k += s[j] * (m * (j + 1) + p * m * (m - 1) // 2)
    return k % G.fr.q


def _entry_count(g, table, n, c):
    """entries of the bucket pipeline for the scalars table[i mod P], i < n: their non-zero digits (the reference's
    partitionScalars, which the engine's digits match).  Below n * W: a signed digit is zero with probability ~2^-c."""
    p = table.shape[0]
    mult = np.maximum((n - np.arange(p, dtype=np.int64) + p - 1) // p, 0)      # how often table row k occurs
    total = 0
    for a in range(0, p, 1 << 17):
        nonzero = (cref.partition_scalars(g, table[a : a + (1 << 17)], c) != 0).sum(axis=0).astype(np.int64)
        total += int((nonzero * mult[a : a + (1 << 17)]).sum())
    return total


def _msm_on_generated_bases(g, n, c, table):
    """bases [i+1]B on the device (spot-checked against the oracle), scalars table[i mod len(table)]; returns (engine c, W, jac)"""
    import torch

    pkg = _pkg()
    G = O.GROUPS[g]
    base = G.encode_affine([G.scalar_mul(G.gen, 0xC0FFEE)])[0]
    w = base.size
    eng = pkg.Engine(g, n, c=c)
    d_pts = d_tab = d_s = None
    try:
        if c:
            assert eng.c == c
        assert eng.nwin == _nwin(g, eng.c)
        assert n * eng.nwin < ENTRY_LIMIT
        entries = _entry_count(g, table, n, eng.c)
        assert entries > (1 << 31), (n, eng.c, eng.nwin, entries)
        d_pts = eng.generate_multiples(base, 1, n)
        j_hi = min(HI_SLOT // n, eng.nwin - 1)          # the point whose window-j_hi digit and rank sit at slot HI_SLOT
        for i in sorted({0, 1, n // 2, n - 2, n - 1, HI_SLOT - j_hi * n}):
            got = d_pts[i * w : (i + 1) * w].cpu().numpy().view(np.uint64)
            assert np.array_equal(got, cref.scalar_mul(g, base, i + 1)), i
        d_tab = eng.to_device(table)
        d_s = d_tab.repeat(-(-n // table.shape[0]), 1)[:n]
        jac = eng.msm_host_result(d_pts, d_s, n)
        return eng.c, eng.nwin, jac, base
    finally:
        eng.close()
        d_pts = d_tab = d_s = None
        torch.cuda.synchronize()
        torch.cuda.empty_cache()


def _assert_point(g, jac, base, k):
    G = O.GROUPS[g]
    w = base.size // 2
    assert np.array_equal(jac[2 * w :], np.array(G.K.encode(G.K.one), dtype=np.uint64))     # output convention: Z = One
    assert np.array_equal(jac[: 2 * w], cref.scalar_mul(g, base, k))


# (group, c (0 = the width model's choice), n); the entries (non-zero digits) come to 1.096 .. 1.125 * 2^31.  At c = 2 and 3 a
# quarter and an eighth of the digits are zero, so those cases need n * W of 1.47 and 1.26 * 2^31 to get there.  K1's mode
# follows k_skew_probe: c <= 3 puts one digit value on more than 1/32 of the sample (rank mode), c >= 8 with uniform scalars stays
# in plain mode.
CASES = [
    pytest.param("bn254_g1", 0, 3 << 26, id="A-bn254_g1-model-plain"),           # model: c = 22, W = 12; split scatter, 2 accumulate launches
    pytest.param("bls12381_g1", 8, 73_819_751, id="C1-bls12381_g1-c8-plain"),    # 12-limb field
    pytest.param("bn254_g2", 3, 31_761_103, id="C2-bn254_g2-c3-rank"),           # Fp2
    pytest.param("secp256k1_g1", 16, 147_639_501, id="C3-secp256k1_g1-c16-plain"),   # full-width moduli, 17-bit last window
    pytest.param("bw6761_g1", 2, 16_664_775, id="C4-bw6761_g1-c2-rank"),         # 24 limbs, 48-byte scalars, lane-parallel tail
    pytest.param("bls24315_g1", 3, 31_761_103, id="C5-bls24315_g1-c3-rank"),     # 10 limbs, 8-byte granules
]


@pytest.mark.parametrize("g,c,n", CASES)
def test_msm_past_2_31_entries(g, c, n):
    L = _native().lib()
    _require_memory(g, n, c or L.gmsm_choose_window_bits(_mx().CURVES[g], n))
    G = O.GROUPS[g]
    table = cref.random_scalars(g, P, 0x5CA1E + n)
    _, _, jac, base = _msm_on_generated_bases(g, n, c, table)
    _assert_point(g, jac, base, _expected_scalar(G, table, n))


def test_msm_at_the_largest_accepted_entry_count():
    """bn254 G1 at c = 2 (W = 127), n = 33,818,637: n * W = 4,294,966,899, the largest count a context accepts.  Every scalar is
    k0 = sum_{j <= 126} 4^j (bits 0, 2, ..., 252), whose 127 digits at c = 2 are all non-zero, so M = n * W entries exactly; with
    K = 256 the last chunk starts at 4,294,966,784 and ends 256 below 2^32.  All entries of a window share one bucket (rank mode,
    the deepest carry join).  Expected: [k0 * n (n + 1) / 2 mod r] B."""
    g, c, n = "bn254_g1", 2, 33_818_637
    assert n * _nwin(g, c) == 4_294_966_899 < ENTRY_LIMIT <= (n + 1) * _nwin(g, c)
    _require_memory(g, n, c)
    G = O.GROUPS[g]
    k0 = sum(4**j for j in range(127))
    enc = G.encode_scalars([k0])
    assert k0 < G.fr.q and np.all(cref.partition_scalars(g, enc, c) != 0)
    _, W, jac, base = _msm_on_generated_bases(g, n, c, enc)
    assert W == 127
    _assert_point(g, jac, base, k0 * (n * (n + 1) // 2) % G.fr.q)


def test_context_refuses_one_past_the_entry_limit():
    pkg = _pkg()
    with pytest.raises(pkg.MultiExpError, match="32-bit entry index"):
        pkg.Engine("bn254_g1", 33_818_638, c=2)


@pytest.mark.parametrize("g,c", [("bn254_g1", 24), ("bls24315_g1", 23)])
def test_widest_windows(g, c):
    """c = 23 and 24, the widths the chooser falls back to when nothing narrower fits the entry index (bn254 G1 from n ~ 3.6e8),
    on a small MultiExp: [sum (i+1) s_i] B over device-generated bases"""
    import torch

    pkg = _pkg()
    n = (1 << 16) + 3
    _require_memory(g, n, c)
    G = O.GROUPS[g]
    base = G.encode_affine([G.scalar_mul(G.gen, 0xC0FFEE)])[0]
    s = cref.random_scalars(g, n, 23 + c)
    eng = pkg.Engine(g, n, c=c)
    try:
        assert eng.c == c
        jac = eng.msm_host_result(eng.generate_multiples(base, 1, n), eng.to_device(s), n)
    finally:
        eng.close()
        torch.cuda.empty_cache()
    _assert_point(g, jac, base, cref.dot_index(g, s, 1))


def test_table_msm_refuses_row_stride_past_the_table_index():
    """gmsm_ctx_msm_tables_device on a small window-table context returns GMSM_EINVAL for row_stride * W >= 2,147,483,000 before
    it enqueues anything: the output stays untouched and no kernel is counted.  The scalars are zero, so no call here reads the
    table, and the largest accepted row stride runs and gives infinity."""
    import torch

    pkg = _pkg()
    g, c, n = "bn254_g1", 8, 16
    eng = pkg.Engine(g, n, c=c, tables=True)
    try:
        W = eng.nwin
        ok = (TABLE_LIMIT - 1) // W
        d_tab = torch.zeros(W * n * 2 * eng.w, dtype=torch.int64, device="cuda")
        d_s = torch.zeros(n * eng.sw, dtype=torch.int64, device="cuda")
        eng._out.fill_(-1)
        with pytest.raises(pkg.MultiExpError, match="31-bit table index"):
            eng.msm_tables(d_tab, ok + 1, d_s, n)
        torch.cuda.synchronize()
        assert bool((eng._out == -1).all()) and eng.last_launches == 0
        out = eng.msm_tables(d_tab, ok, d_s, n).cpu().numpy()
        assert not out.any() and eng.last_launches > 0
        launches = eng.last_launches
        eng._out.fill_(-1)
        with pytest.raises(pkg.MultiExpError, match="31-bit table index"):
            eng.msm_tables(d_tab, ok + 1, d_s, n)
        torch.cuda.synchronize()
        assert bool((eng._out == -1).all()) and eng.last_launches == launches
    finally:
        eng.close()

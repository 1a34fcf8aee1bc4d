"""The two 32-bit index limits of the bucket pipeline, checked on the host side (no GPU needed).

* A context numbers its bucket entries with 32-bit indices: it accepts n with n * W < 4,294,967,000 (W = number of windows), so
  the window chooser must return a width that fits whenever one exists.
* A window table entry is (j * row_stride + i) << 1 | sign in 32 bits: tables need row_stride * W < 2,147,483,000.

The device side of both limits (a MultiExp at the largest accepted n * W, the refusals of a live context) is in
tests/test_gpu_scale_limits.py."""
import importlib

ENTRY_LIMIT = 4_294_967_000
TABLE_LIMIT = 2_147_483_000
GROUPS = range(13)


def _native():
    return importlib.import_module("gnark-crypto_b200._native")


def _bits(cid):
    return importlib.import_module("gnark-crypto_b200.multiexp").SCALAR_BITS[cid]


def _nwin(bits, c):
    return (bits + c - 1) // c


def _grid(bits):
    """powers of two up to 2^31 - 1, the band [3.5e8, 4e8] every 10^5, and both sides of each width's entry limit"""
    ns = {(1 << k) for k in range(4, 31)} | {(1 << 31) - 1}
    ns |= set(range(350_000_000, 400_000_001, 100_000))
    for c in range(2, 25):
        edge = -(-ENTRY_LIMIT // _nwin(bits, c))        # smallest n that no longer fits width c
        ns |= {edge - 1, edge, edge + 1}
    return sorted(n for n in ns if 1 <= n < (1 << 31))


def test_chooser_returns_a_width_that_fits_the_entry_index():
    """gmsm_choose_window_bits (and with it Engine(c=0), dist.window_bits_for_total and the host entry points) must not pick a
    width whose n * W a context refuses while a width in [2, 24] would be accepted"""
    L = _native().lib()
    bad = []
    for cid in GROUPS:
        bits = _bits(cid)
        for n in _grid(bits):
            fitting = [c for c in range(2, 25) if n * _nwin(bits, c) < ENTRY_LIMIT]
            c = L.gmsm_choose_window_bits(cid, n)
            assert 2 <= c <= 24, (cid, n, c)
            if fitting and c not in fitting:
                bad.append((cid, n, c, fitting[0]))
    assert not bad, "%d choices refused by the context, e.g. (group, n, chosen, smallest fitting) %s" % (len(bad), bad[:5])


def test_chooser_takes_c24_where_only_it_fits():
    """bn254 G1 (254-bit scalars): c <= 23 means W >= 12, so from n = 357,913,917 (= ceil(4,294,967,000 / 12)) up to
    390,451,545 (the last n with 11 n below the limit) only c = 24 (W = 11) fits; below that band the model's c = 22 stays"""
    L = _native().lib()
    assert L.gmsm_choose_window_bits(0, 357_913_916) == 22
    for n in (357_913_917, 375_000_000, 390_451_545):
        assert L.gmsm_choose_window_bits(0, n) == 24, n
    assert 12 * 357_913_917 >= ENTRY_LIMIT > 11 * 390_451_545


def test_table_build_refuses_row_stride_past_the_table_index():
    """gmsm_tables_build_device checks row_stride * W < 2,147,483,000 before it touches a device: with n = 0 and null pointers
    the largest accepted row stride returns GMSM_OK and the next one GMSM_EINVAL, for every group and several widths"""
    nat = _native()
    L = nat.lib()
    for cid in GROUPS:
        bits = _bits(cid)
        for c in (2, 3, 8, 13, 16, 22, 24):
            W = _nwin(bits, c)
            ok = (TABLE_LIMIT - 1) // W
            assert ok * W < TABLE_LIMIT <= (ok + 1) * W
            assert L.gmsm_tables_build_device(cid, c, None, 0, None, ok, None) == nat.GMSM_OK, (cid, c)
            assert L.gmsm_tables_build_device(cid, c, None, 0, None, ok + 1, None) == nat.GMSM_EINVAL, (cid, c)
            assert "31-bit table index" in nat.last_error(), (cid, c, nat.last_error())

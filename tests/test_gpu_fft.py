"""Next-row N3: the GPU Fr FFT against the oracle (small sizes, all decimation / coset / inverse variants,
both scalar fields, custom shift) and size-independent properties at 2^20 / 2^22 (round trips, the DIF+DIT
compositions gnark uses, evaluation of a sparse polynomial in closed form)."""
import importlib
import random

import numpy as np
import pytest

from oracle import oracle as O

pytestmark = pytest.mark.gpu
FR = {"bn254": "bn254_fr", "bls12381": "bls12381_fr", "bls12377": "bls12377_fr"}


def _fft():
    import gnark_crypto_b200  # noqa: F401

    return importlib.import_module("gnark-crypto_b200.fft")


def _enc(f, vals):
    return np.array([f.to_limbs(f.to_mont(v)) for v in vals], dtype=np.uint64)


def _dec(f, arr):
    return [f.from_mont(O.Field.from_limbs([int(x) for x in r])) for r in arr]


@pytest.mark.parametrize("curve", ["bn254", "bls12381", "bls12377"])
@pytest.mark.parametrize("logn", [0, 1, 2, 5, 10, 11, 13])
def test_fft_matches_oracle(curve, logn):
    fft = _fft()
    f = O.FIELDS[FR[curve]]
    n = 1 << logn
    rng = random.Random(logn)
    vals = [rng.randrange(f.q) for _ in range(n)]
    od = O.FFTDomain(FR[curve], n)
    d = fft.NewDomain(curve, n)
    assert d.Cardinality == n
    assert _dec(f, np.stack([d.Generator, d.GeneratorInv, d.CardinalityInv, d.FrMultiplicativeGen, d.FrMultiplicativeGenInv])) == [
        od.generator, od.generator_inv, od.cardinality_inv, od.shift, od.shift_inv]
    for dec in (O.DIT, O.DIF):
        for coset in (False, True):
            a = _enc(f, vals)
            assert _dec(f, d.FFT(a, dec, OnCoset=coset)) == od.fft(vals, dec, coset), (dec, coset)
            a = _enc(f, vals)
            assert _dec(f, d.FFTInverse(a, dec, OnCoset=coset)) == od.fft_inverse(vals, dec, coset), (dec, coset)
    d.close()


def _edge_inputs(f, n):
    """Fr vectors at the edges of the Montgomery arithmetic (plain values; _enc stores value * R mod q)"""
    q = f.q
    raw_qm1 = (q - 1) * f.Rinv % q                                  # stored limbs q - 1
    return {
        "all_q-1": [q - 1] * n,
        "all_limbs_q-1": [raw_qm1] * n,
        "alternating_0_q-1": [0 if i % 2 == 0 else q - 1 for i in range(n)],
        "alternating_limbs": [raw_qm1 if i % 2 == 0 else 0 for i in range(n)],
        "powers_of_two": [(1 << (i % f.bits)) % q for i in range(n)],
    }


@pytest.mark.parametrize("curve", ["bn254", "bls12381", "bls12377"])
@pytest.mark.parametrize("logn", [10, 11, 14])
def test_fft_edge_inputs(curve, logn):
    """extreme Fr inputs through the device FFT at one tile (2^10), one global stage (2^11) and four global stages (2^14):
    FFT and FFTInverse, DIT and DIF, plain and on the coset, in full against the oracle; then the same on a domain whose
    coset shift is q - 1"""
    fft = _fft()
    f = O.FIELDS[FR[curve]]
    n = 1 << logn
    od = O.FFTDomain(FR[curve], n)
    d = fft.NewDomain(curve, n)
    od_m1 = O.FFTDomain(FR[curve], n, shift=f.q - 1)
    d_m1 = fft.NewDomain(curve, n, shift=_enc(f, [f.q - 1])[0])
    try:
        for name, vals in _edge_inputs(f, n).items():
            for dec in (O.DIT, O.DIF):
                for coset in (False, True):
                    assert _dec(f, d.FFT(_enc(f, vals), dec, OnCoset=coset)) == od.fft(vals, dec, coset), (name, dec, coset)
                    assert _dec(f, d.FFTInverse(_enc(f, vals), dec, OnCoset=coset)) == od.fft_inverse(vals, dec, coset), (name, dec, coset)
                if name in ("all_q-1", "alternating_0_q-1"):
                    assert _dec(f, d_m1.FFT(_enc(f, vals), dec, OnCoset=True)) == od_m1.fft(vals, dec, True), (name, dec, "shift q-1")
                    assert _dec(f, d_m1.FFTInverse(_enc(f, vals), dec, OnCoset=True)) == od_m1.fft_inverse(vals, dec, True), (name, dec, "shift q-1")
    finally:
        d.close()
        d_m1.close()


def test_fft_custom_shift_and_errors():
    fft = _fft()
    f = O.FIELDS["bn254_fr"]
    n = 64
    vals = list(range(1, n + 1))
    shift = 987654321
    d = fft.NewDomain("bn254", n - 3, shift=_enc(f, [shift])[0])     # cardinality = next power of two
    od = O.FFTDomain("bn254_fr", n, shift=shift)
    a = _enc(f, vals)
    assert _dec(f, d.FFT(a, O.DIF, OnCoset=True)) == od.fft(vals, O.DIF, True)
    with pytest.raises(Exception, match="cardinality"):
        d.FFT(_enc(f, vals[:32]), O.DIF)
    with pytest.raises(Exception, match="too big"):
        fft.NewDomain("bn254", 1 << 29)                              # bn254 fr: maxOrderRoot = 28
    d.close()


@pytest.mark.parametrize("curve,logn", [("bn254", 20), ("bn254", 22), ("bls12381", 20)])
def test_fft_large_properties(curve, logn):
    import torch

    fft = _fft()
    f = O.FIELDS[FR[curve]]
    n = 1 << logn
    d = fft.NewDomain(curve, n)
    rng = np.random.default_rng(logn)
    a = rng.integers(0, 2**62, size=(n, 4), dtype=np.uint64)
    a[:, 3] &= np.uint64((1 << 59) - 1)                             # < q, arbitrary Montgomery residues
    da = torch.from_numpy(a.view(np.int64)).cuda()
    orig = da.clone()
    # FFT(DIF) then FFTInverse(DIT) is the identity without any bit reversal (the pattern gnark's provers use)
    d.fft_device(da, False, O.DIF)
    assert not torch.equal(da, orig)
    d.fft_device(da, True, O.DIT)
    assert torch.equal(da, orig)
    # same on the coset, and the other composition through explicit bit reversals
    d.fft_device(da, False, O.DIF, coset=True)
    d.fft_device(da, True, O.DIT, coset=True)
    assert torch.equal(da, orig)
    d.bit_reverse_device(da)
    d.fft_device(da, False, O.DIT)
    d.fft_device(da, True, O.DIF)
    d.bit_reverse_device(da)
    assert torch.equal(da, orig)
    # closed form: p(X) = c0 + c1 X^k  ->  evaluations c0 + c1 w^(k i); check a few positions (DIT: natural output)
    k, c0, c1 = 12345, 7, 11
    vals = np.zeros((n, 4), dtype=np.uint64)
    vals[0] = _enc(f, [c0])[0]
    vals[k] = _enc(f, [c1])[0]
    dv = torch.from_numpy(vals.view(np.int64)).cuda()
    d.bit_reverse_device(dv)
    d.fft_device(dv, False, O.DIT)
    out = dv.cpu().numpy().view(np.uint64)
    od = O.FFTDomain(FR[curve], n)
    for i in (0, 1, 2, 1000, n // 2 + 3, n - 1):
        want = (c0 + c1 * pow(od.generator, k * i, f.q)) % f.q
        assert _dec(f, out[i : i + 1])[0] == want, i
    d.close()

"""Shared op-level test vectors: element-wise field / point operations checked against the oracle.
Used by tests/test_hostcheck.py (CPU build of the arithmetic headers) and tests/test_gpu_ops.py
(the same operations executed by the sm_100a device code)."""
import random

import numpy as np

from oracle import oracle as O

OPS = dict(FMUL=0, FADD=1, FSUB=2, FSQR=3, FNEG=4, FDBL=5, FINV=6, ADD_MIXED=7, SUB_MIXED=8, ADD=9, DOUBLE=10, TO_AFFINE=11,
           FR_FROM_MONT=12, DOT2=13, FP_DOT4=14)


def u32(a):
    return np.ascontiguousarray(a, dtype=np.uint64).view(np.uint32).reshape(a.shape[0], -1)


def enc_f(G, vals):
    return np.array([G.K.encode(v) for v in vals], dtype=np.uint64)


def dec_f(G, arr):
    arr = np.ascontiguousarray(arr, dtype=np.uint32).view(np.uint64)
    return [G.K.decode([int(x) for x in r]) for r in arr]


def enc_xyzz(G, pts):
    return np.array([sum((G.K.encode(c) for c in p), []) for p in pts], dtype=np.uint64)


def dec_xyzz(G, arr):
    arr = np.ascontiguousarray(arr, dtype=np.uint32).view(np.uint64)
    w = G.K.words
    return [[G.K.decode([int(x) for x in r[i * w : (i + 1) * w]]) for i in range(4)] for r in arr]


def field_values(G, rng, n):
    q = G.K.q
    f = G.K.f
    specials = [0, 1, q - 1, q - 2, f.Rmod, f.R2, (q - 1) // 2, (1 << (f.bits - 1)) % q, 0xFFFFFFFF, 1 << 32, (1 << 64) - 1]
    vals = specials + [rng.randrange(q) for _ in range(n)]
    if G.K.ext == 1:
        return vals
    return [(a, b) for a, b in zip(vals, reversed(vals))] + [(0, 0), (1, 0), (0, 1), (q - 1, q - 1)]


def random_xyzz(G, rng, k, z=None):
    """a non-trivial extended-Jacobian representation of [k]G: (x z^2, y z^3, z^2, z^3), z random unless given"""
    K = G.K
    a = G.scalar_mul(G.gen, k)
    if G.aff_is_inf(a):
        return G.xyzz_inf()
    if z is None:
        z = K.from_int(rng.randrange(1, K.q)) if K.ext == 1 else (rng.randrange(1, K.q), rng.randrange(K.q))
    return xyzz_with_z(G, a, z)


def xyzz_with_z(G, a, z):
    """the extended-Jacobian representation (x z^2, y z^3, z^2, z^3) of the finite affine point a"""
    K = G.K
    zz = K.sqr(z)
    zzz = K.mul(zz, z)
    return [K.mul(a[0], zz), K.mul(a[1], zzz), zz, zzz]


def check_field_ops(G, run):
    """run(op, a_u32, b_u32 or None, out_words) -> u32 array"""
    K = G.K
    rng = random.Random(11)
    a = field_values(G, rng, 40)
    b = list(reversed(a))
    A, B = u32(enc_f(G, a)), u32(enc_f(G, b))
    w32 = 2 * K.words
    assert dec_f(G, run(OPS["FMUL"], A, B, w32)) == [K.mul(x, y) for x, y in zip(a, b)]
    assert dec_f(G, run(OPS["FADD"], A, B, w32)) == [K.add(x, y) for x, y in zip(a, b)]
    assert dec_f(G, run(OPS["FSUB"], A, B, w32)) == [K.sub(x, y) for x, y in zip(a, b)]
    assert dec_f(G, run(OPS["FSQR"], A, None, w32)) == [K.sqr(x) for x in a]
    assert dec_f(G, run(OPS["FNEG"], A, None, w32)) == [K.neg(x) for x in a]
    assert dec_f(G, run(OPS["FDBL"], A, None, w32)) == [K.dbl(x) for x in a]
    assert dec_f(G, run(OPS["FINV"], A[:12], None, w32)) == [K.inv(x) for x in a[:12]]
    # outputs are fully reduced Montgomery limbs: re-encoding the decoded value reproduces the bytes
    out = run(OPS["FMUL"], A, B, w32)
    assert np.array_equal(u32(enc_f(G, dec_f(G, out))), out)


def check_fr_from_mont(G, run):
    fr = G.fr
    rng = random.Random(5)
    vals = [0, 1, fr.q - 1, fr.Rmod] + [rng.randrange(fr.q) for _ in range(30)]
    A = u32(np.array([fr.to_limbs(v) for v in vals], dtype=np.uint64))
    out = run(OPS["FR_FROM_MONT"], A, None, 2 * fr.limbs)
    got = [O.Field.from_limbs([int(x) for x in r]) for r in np.ascontiguousarray(out).view(np.uint64)]
    assert got == [fr.from_mont(v) for v in vals]


def check_point_ops(G, run):
    K = G.K
    rng = random.Random(23)
    w32 = 2 * K.words
    ks = [1, 2, 3, 5, 7, 11, 100, G.fr.q - 1, G.fr.q - 2, rng.randrange(G.fr.q), rng.randrange(G.fr.q)]
    # (p, a) pairs: generic, p = inf, a = inf, p == a (doubling), p == -a (cancellation)
    ps, as_ = [], []
    for k1 in ks[:8]:
        for k2 in (1, 2, 5, k1, (G.fr.q - k1) % G.fr.q):
            ps.append(random_xyzz(G, rng, k1))
            as_.append(G.scalar_mul(G.gen, k2))
    ps.append(G.xyzz_inf()); as_.append(G.scalar_mul(G.gen, 9))
    ps.append([K.zero, K.zero, K.zero, K.zero]); as_.append(G.scalar_mul(G.gen, 9))  # all-zero infinity (memset buckets)
    ps.append(random_xyzz(G, rng, 9)); as_.append(G.aff_inf())
    ps.append(G.xyzz_inf()); as_.append(G.aff_inf())
    P, A = u32(enc_xyzz(G, ps)), u32(G.encode_affine(as_))
    for op, neg in (("ADD_MIXED", False), ("SUB_MIXED", True)):
        got = dec_xyzz(G, run(OPS[op], P, A, 4 * w32))
        for p, a, g in zip(ps, as_, got):
            want = G.add_mixed(list(p), a, negate=neg)
            assert G.xyzz_to_affine(g) == G.xyzz_to_affine(want)
            if not K.is_zero(want[2]):
                assert g == want  # the exact coordinates of the reference's formulas (g1.go:822-930)
    # full add / double
    qs = [random_xyzz(G, rng, k) for k in (1, 2, 5)] * (len(ps) // 3 + 1)
    qs = qs[: len(ps)]
    qs[0] = list(ps[0])                     # same representation -> doubling branch
    k0 = ks[1]
    ps[1], qs[1] = random_xyzz(G, rng, k0), random_xyzz(G, rng, k0)        # same point, different z -> doubling
    ps[2], qs[2] = random_xyzz(G, rng, k0), random_xyzz(G, rng, G.fr.q - k0)  # opposite -> infinity
    qs[3] = G.xyzz_inf()
    P, Q = u32(enc_xyzz(G, ps)), u32(enc_xyzz(G, qs))
    got = dec_xyzz(G, run(OPS["ADD"], P, Q, 4 * w32))
    for p, q, g in zip(ps, qs, got):
        want = G.xyzz_add(list(p), list(q))
        assert G.xyzz_to_affine(g) == G.xyzz_to_affine(want)
        if not K.is_zero(want[2]) and not K.is_zero(p[2]):
            assert g == want
    got = dec_xyzz(G, run(OPS["DOUBLE"], P, None, 4 * w32))
    for p, g in zip(ps, got):
        assert G.xyzz_to_affine(g) == G.xyzz_to_affine(G.xyzz_double(p))
    # normalisation: byte-exact affine normal form
    got = run(OPS["TO_AFFINE"], P[:10], None, 2 * w32)
    want = u32(G.encode_affine([G.xyzz_to_affine(p) for p in ps[:10]]))
    assert np.array_equal(got, want)


# ------------------------------------------------------------------------------------------
# Extreme operands.  The Montgomery routines go wrong at inputs random operands almost never reach: limbs of all ones or of
# the modulus' own value, single bits, results in [q, 2q) that differ from q only in the low limbs.  The expected values of
# check_field_edges are computed on the raw Montgomery limbs with plain integers (x y R^-1 mod q, not the oracle's Field
# methods), so the vectors are checked against big-integer arithmetic and nothing else.
# ------------------------------------------------------------------------------------------
def extreme_values(f):
    """reduced raw limb values (< q) of field f at the edges of the limb arithmetic, without duplicates"""
    q, nl = f.q, 2 * f.limbs
    vals = [0, 1, 2, q - 1, q - 2, f.Rmod, f.R2, (q - 1) // 2, (q + 1) // 2]
    for k in range(0, 32 * nl, 7):
        vals += [(1 << k) % q, ((1 << k) - 1) % q, (q - (1 << k)) % q]
    top = (1 << (32 * nl)) - 1
    for k in range(nl):
        vals.append((top ^ (0xFFFFFFFF << (32 * k))) % q)
        vals.append((0xFFFFFFFF << (32 * k)) % q)
    # the top limb equal to q's: q's top limb alone, with all-ones or q's own limbs below (minus one limb), and each limb of q alone
    qtop = q >> (32 * (nl - 1)) << (32 * (nl - 1))
    vals += [qtop, (qtop | ((1 << (32 * (nl - 1))) - 1)) % q, qtop - 1]
    for k in range(nl):
        vals.append(q & (0xFFFFFFFF << (32 * k)))
        vals.append(q - (1 << (32 * k)))
    vals = [v % q for v in vals]
    return list(dict.fromkeys(vals))


def extreme_values_fp2(f, rng, n_random):
    """Fp2 raw limb pairs: the cross product of a reduced extreme set, plus random pairs"""
    q, nl = f.q, 2 * f.limbs
    qtop = q >> (32 * (nl - 1)) << (32 * (nl - 1))
    small = [0, 1, 2, q - 1, q - 2, f.Rmod, f.R2, (q - 1) // 2, (q + 1) // 2, qtop, q - (1 << 32), ((1 << (32 * nl)) - 1) % q,
             (1 << (32 * (nl - 1))) - 1, 0xFFFFFFFF]
    small = list(dict.fromkeys(v % q for v in small))
    return [(a, b) for a in small for b in small] + [(rng.randrange(q), rng.randrange(q)) for _ in range(n_random)]


def _ints_u32(vals, nl):
    """raw integers -> (n, nl) little-endian u32 limb rows"""
    return np.frombuffer(b"".join(v.to_bytes(4 * nl, "little") for v in vals), dtype=np.uint32).reshape(len(vals), nl).copy()


def _u32_ints(arr):
    arr = np.ascontiguousarray(arr, dtype=np.uint32)
    return [int.from_bytes(r.tobytes(), "little") for r in arr]


class RawField:
    """expected values on raw Montgomery limbs (stored integer x stands for x R^-1) with plain integers: Fp (ext 1) or
    Fp2 = Fp[u] / (u^2 - beta) (ext 2, elements as pairs).  R = 2^(32 * limbs) for the 32-bit limb count of the field."""

    def __init__(self, q, nl, ext, beta=None):
        self.q, self.nl, self.ext, self.beta = q, nl, ext, beta
        self.R = 1 << (32 * nl)
        self.Rinv = pow(self.R, -1, q)
        self.R2 = self.R * self.R % q

    # base field
    def mul1(self, x, y):
        return x * y * self.Rinv % self.q

    def inv1(self, x):
        return pow(x, -1, self.q) * self.R2 % self.q if x else 0

    # coordinate field
    def _map(self, fn, *xs):
        return fn(*xs) if self.ext == 1 else tuple(fn(*c) for c in zip(*xs))

    def add(self, x, y):
        return self._map(lambda a, b: (a + b) % self.q, x, y)

    def sub(self, x, y):
        return self._map(lambda a, b: (a - b) % self.q, x, y)

    def neg(self, x):
        return self._map(lambda a: -a % self.q, x)

    def dbl(self, x):
        return self._map(lambda a: 2 * a % self.q, x)

    def mul(self, x, y):
        if self.ext == 1:
            return self.mul1(x, y)
        q = self.q
        return ((x[0] * y[0] + self.beta * x[1] * y[1]) * self.Rinv % q, (x[0] * y[1] + x[1] * y[0]) * self.Rinv % q)

    def inv(self, x):
        if self.ext == 1:
            return self.inv1(x)
        # (x0 - x1 u) / (x0^2 - beta x1^2): on raw limbs the R factors leave x_k R^2 / d
        q = self.q
        d = (x[0] * x[0] - self.beta * x[1] * x[1]) % q
        di = pow(d, -1, q) * self.R2 % q if d else 0
        return (x[0] * di % q, -x[1] * di % q)

    def dot2(self, x, y, u, v):
        return self.add(self.mul(x, y), self.mul(u, v))

    def dot4(self, xs, ys):
        return sum(x * y for x, y in zip(xs, ys)) * self.Rinv % self.q

    # memory
    def enc(self, vals):
        if self.ext == 1:
            return _ints_u32(vals, self.nl)
        return _ints_u32([a | b << (32 * self.nl) for a, b in vals], 2 * self.nl)

    def dec(self, arr):
        """output rows -> elements; every component must be canonical (< q)"""
        ints = _u32_ints(arr)
        if self.ext == 1:
            out = ints
            comps = ints
        else:
            m = (1 << (32 * self.nl)) - 1
            out = [(v & m, v >> (32 * self.nl)) for v in ints]
            comps = [c for p in out for c in p]
        bad = [i for i, c in enumerate(comps) if c >= self.q]
        assert not bad, "non-canonical output limbs (>= q) at component %d of %d" % (bad[0], len(comps))
        return out


def raw_field(G):
    f = G.K.f
    return RawField(f.q, 2 * f.limbs, G.K.ext, getattr(G.K, "beta", None))


def _expect(got, want, what):
    bad = [i for i, (g, w) in enumerate(zip(got, want)) if g != w]
    assert len(got) == len(want) and not bad, "%s: %d of %d wrong, first at %d" % (what, len(bad), len(want), bad[0] if bad else -1)


def _rotations(n, n_perm, rng):
    """n_perm rotation offsets of a list of n (None: all n, i.e. every element against every other)"""
    if n_perm is None or n_perm >= n:
        return list(range(n))
    return [0, 1] + rng.sample(range(2, n), n_perm - 2) if n_perm > 2 else list(range(n_perm))


def check_field_edges(G, run, n_random, n_perm=None, seed=29):
    """the coordinate-field ops, the fused sums of products (DOT2 in the coordinate field, FP_DOT4 in the base field) and the
    inversion at extreme operands: every extreme value against n_perm rotations of the extreme list (None: all of them),
    plus n_random random operands; for the Fp2 groups additionally the base-field extremes through FP_DOT4.
    run(op, a_u32, b_u32 or None, out_words) -> u32 array"""
    F = raw_field(G)
    B = RawField(F.q, F.nl, 1)
    q = F.q
    rng = random.Random(seed)
    ext = extreme_values(G.K.f)
    if F.ext == 1:
        E = ext
        rnd = lambda: rng.randrange(q)
        qm1 = q - 1
    else:
        E = extreme_values_fp2(G.K.f, rng, 40)
        rnd = lambda: (rng.randrange(q), rng.randrange(q))
        qm1 = (q - 1, q - 1)
    fw = F.nl * F.ext
    rots = _rotations(len(E), n_perm, rng)
    a = [E[i] for _ in rots for i in range(len(E))] + [rnd() for _ in range(n_random)] + [qm1]
    b = [E[(i + r) % len(E)] for r in rots for i in range(len(E))] + [rnd() for _ in range(n_random)] + [qm1]
    A, Bm = F.enc(a), F.enc(b)
    _expect(F.dec(run(OPS["FMUL"], A, Bm, fw)), [F.mul(x, y) for x, y in zip(a, b)], "FMUL")
    _expect(F.dec(run(OPS["FADD"], A, Bm, fw)), [F.add(x, y) for x, y in zip(a, b)], "FADD")
    _expect(F.dec(run(OPS["FSUB"], A, Bm, fw)), [F.sub(x, y) for x, y in zip(a, b)], "FSUB")
    _expect(F.dec(run(OPS["FSQR"], A, None, fw)), [F.mul(x, x) for x in a], "FSQR")
    _expect(F.dec(run(OPS["FNEG"], A, None, fw)), [F.neg(x) for x in a], "FNEG")
    _expect(F.dec(run(OPS["FDBL"], A, None, fw)), [F.dbl(x) for x in a], "FDBL")
    _expect(F.dec(run(OPS["FINV"], F.enc(E), None, fw)), [F.inv(x) for x in E], "FINV")
    # x y + u v: y, u, v from further rotations of the extremes
    u = [E[(i + 2 * r + 1) % len(E)] for r in rots for i in range(len(E))] + [rnd() for _ in range(n_random)] + [qm1]
    v = [E[(i + 3 * r + 2) % len(E)] for r in rots for i in range(len(E))] + [rnd() for _ in range(n_random)] + [qm1]
    got = F.dec(run(OPS["DOT2"], np.hstack([A, F.enc(u)]), np.hstack([Bm, F.enc(v)]), fw))
    _expect(got, [F.dot2(*t) for t in zip(a, b, u, v)], "DOT2")
    # four base-field products: x_k and y_k from eight rotations of the base-field extremes
    n = len(ext)
    brots = _rotations(n, n_perm, rng)
    xs = [[ext[(i + (2 * k + 1) * r + k) % n] for r in brots for i in range(n)] for k in range(4)]
    ys = [[ext[(i + (2 * k + 2) * r + 3 * k) % n] for r in brots for i in range(n)] for k in range(4)]
    for k in range(4):
        xs[k] += [rng.randrange(q) for _ in range(n_random)] + [q - 1]
        ys[k] += [rng.randrange(q) for _ in range(n_random)] + [q - 1]
    got = B.dec(run(OPS["FP_DOT4"], np.hstack([B.enc(c) for c in xs]), np.hstack([B.enc(c) for c in ys]), B.nl))
    _expect(got, [B.dot4(x, y) for x, y in zip(zip(*xs), zip(*ys))], "FP_DOT4")


def z_edges(G):
    """z coordinates at the edges of the field for the extended-Jacobian inputs of check_point_edges"""
    K, f = G.K, G.K.f
    q = f.q
    zs = [1, 2, q - 1, 1 << 32, 1 << 64, 1 << (f.bits - 2), f.Rmod, f.Rinv, (q - 1) // 2]
    if K.ext == 1:
        return zs
    return [(z, 0) for z in zs] + [(0, z) for z in zs] + [(q - 1, q - 1)]


def check_point_edges(G, run):
    """the point formulas on extended-Jacobian inputs whose z is chosen at the edges of the field (z_edges), exact coordinates
    against the oracle's formulas"""
    K = G.K
    w32 = 2 * K.words
    zs = z_edges(G)
    r = G.fr.q
    mult = {k: G.scalar_mul(G.gen, k) for k in (1, 5, 3, 7, r - 2, 100, r - 3, r - 7, 2, r - 100)}
    ps, as_, qs = [], [], []
    for i, z in enumerate(zs):
        k = (3, 7, r - 2, 100)[i % 4]
        for j, k2 in enumerate((1, 5, k, r - k)):     # generic, generic, doubling, cancellation
            ps.append(xyzz_with_z(G, mult[k], z))
            as_.append(mult[k2])
            qs.append(xyzz_with_z(G, mult[k2], zs[(i + j + 1) % len(zs)]))
    P, A, Q = u32(enc_xyzz(G, ps)), u32(G.encode_affine(as_)), u32(enc_xyzz(G, qs))
    for op, neg in (("ADD_MIXED", False), ("SUB_MIXED", True)):
        got = dec_xyzz(G, run(OPS[op], P, A, 4 * w32))
        for p, a, g in zip(ps, as_, got):
            want = G.add_mixed(list(p), a, negate=neg)
            assert G.xyzz_to_affine(g) == G.xyzz_to_affine(want)
            if not K.is_zero(want[2]):
                assert g == want, op
    got = dec_xyzz(G, run(OPS["ADD"], P, Q, 4 * w32))
    for p, q_, g in zip(ps, qs, got):
        want = G.xyzz_add(list(p), list(q_))
        assert G.xyzz_to_affine(g) == G.xyzz_to_affine(want)
        if not K.is_zero(want[2]):
            assert g == want, "ADD"
    got = dec_xyzz(G, run(OPS["DOUBLE"], P, None, 4 * w32))
    assert got == [G.xyzz_double(p) for p in ps], "DOUBLE"
    got = run(OPS["TO_AFFINE"], P, None, 2 * w32)
    assert np.array_equal(got, u32(G.encode_affine([G.xyzz_to_affine(p) for p in ps]))), "TO_AFFINE"

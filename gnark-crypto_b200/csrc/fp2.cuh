// Quadratic extension Fp2 = Fp[u]/(u^2 - beta) for G2: beta = -1 for bn254 and bls12-381, beta = -5 for
// bls12-377 (P::FP2_NONRES; ecc/bls12-377/internal/fptower/e2_bls377.go:12-80).
//
// Replaces (reference): E2.Mul/Square ecc/bn254/internal/fptower/e2_bn254.go:28-51 (asm
// e2_amd64.s:393,548), Add/Sub/Double/Neg e2.go:104-126, Inverse e2_bn254.go:61-73; identical
// formulas ecc/bls12-381/internal/fptower/e2_bls381.go:16-74.  Memory order A0, A1 (e2.go:14-16).
#pragma once
#include "field.cuh"

namespace gmsm {

template <class P>
struct Fp2 {
  using Params = P;
  static constexpr int N = 2 * P::N;  // 32-bit words in memory
  Fp<P> a0, a1;
  GMSM_HD static Fp2 zero() { return Fp2{Fp<P>::zero(), Fp<P>::zero()}; }
  GMSM_HD static Fp2 one() { return Fp2{Fp<P>::one(), Fp<P>::zero()}; }
  GMSM_HD bool is_zero() const { return a0.is_zero() && a1.is_zero(); }
  GMSM_HD bool operator==(const Fp2& b) const { return a0 == b.a0 && a1 == b.a1; }
  GMSM_HD bool operator!=(const Fp2& b) const { return !(*this == b); }
};

template <class P> struct base_field<Fp2<P>> { using type = Fp<P>; };

template <class P> GMSM_HD Fp2<P> f_add(const Fp2<P>& a, const Fp2<P>& b) { return Fp2<P>{fp_add(a.a0, b.a0), fp_add(a.a1, b.a1)}; }
template <class P> GMSM_HD Fp2<P> f_sub(const Fp2<P>& a, const Fp2<P>& b) { return Fp2<P>{fp_sub(a.a0, b.a0), fp_sub(a.a1, b.a1)}; }
template <class P> GMSM_HD Fp2<P> f_dbl(const Fp2<P>& a) { return Fp2<P>{fp_dbl(a.a0), fp_dbl(a.a1)}; }
template <class P> GMSM_HD Fp2<P> f_neg(const Fp2<P>& a) { return Fp2<P>{fp_neg(a.a0), fp_neg(a.a1)}; }

template <class P>
GMSM_HD Fp<P> fp_mul_by5(const Fp<P>& c) {  // fp.MulBy5
  return fp_add(fp_dbl(fp_dbl(c)), c);
}

#if defined(GMSM_FP2_LAZY)
// Fp2 product with lazy reduction (beta = -1 only): three double-width products, two reductions -- z1 = (x0+x1)(y0+y1) - x0y0 -
// x1y1 and z0 = x0y0 - x1y1 + qR are formed on 2N limbs and reduced once each: 3 N^2 + 2 (N^2 + N) = 336 IMAD.WIDE for N = 8
// against Karatsuba's 3 x 136 = 408.  Same unique reduced values.
template <class P>
GMSM_HD Fp2<P> fp2_mul_lazy_inline(const Fp2<P>& x, const Fp2<P>& y) {
    constexpr int N = P::N;
    uint32_t sx[N], sy[N], T0[2 * N], T1[2 * N], T2[2 * N];
#if defined(GMSM_PTX_PATH)
    sx[0] = add_cc(x.a0.l[0], x.a1.l[0]);
#pragma unroll
    for (int i = 1; i < N - 1; i++) sx[i] = addc_cc(x.a0.l[i], x.a1.l[i]);
    sx[N - 1] = addc(x.a0.l[N - 1], x.a1.l[N - 1]);
    sy[0] = add_cc(y.a0.l[0], y.a1.l[0]);
#pragma unroll
    for (int i = 1; i < N - 1; i++) sy[i] = addc_cc(y.a0.l[i], y.a1.l[i]);
    sy[N - 1] = addc(y.a0.l[N - 1], y.a1.l[N - 1]);
#else
    { uint64_t c = 0; for (int i = 0; i < N; i++) { c += (uint64_t)x.a0.l[i] + x.a1.l[i]; sx[i] = (uint32_t)c; c >>= 32; } }
    { uint64_t c = 0; for (int i = 0; i < N; i++) { c += (uint64_t)y.a0.l[i] + y.a1.l[i]; sy[i] = (uint32_t)c; c >>= 32; } }
#endif
    fp_mul_wide<P>(x.a0.l, y.a0.l, T0);
    fp_mul_wide<P>(x.a1.l, y.a1.l, T1);
    fp_mul_wide<P>(sx, sy, T2);
#if defined(GMSM_PTX_PATH)
    // T2 -= T0; T2 -= T1   (x0 y1 + x1 y0 >= 0: no borrow out)
    T2[0] = sub_cc(T2[0], T0[0]);
#pragma unroll
    for (int i = 1; i < 2 * N - 1; i++) T2[i] = subc_cc(T2[i], T0[i]);
    T2[2 * N - 1] = subc(T2[2 * N - 1], T0[2 * N - 1]);
    T2[0] = sub_cc(T2[0], T1[0]);
#pragma unroll
    for (int i = 1; i < 2 * N - 1; i++) T2[i] = subc_cc(T2[i], T1[i]);
    T2[2 * N - 1] = subc(T2[2 * N - 1], T1[2 * N - 1]);
    // T0 = T0 - T1 + q R  (mod 2^(64N); the true value lies in (qR - q^2, qR + q^2))
    T0[0] = sub_cc(T0[0], T1[0]);
#pragma unroll
    for (int i = 1; i < 2 * N - 1; i++) T0[i] = subc_cc(T0[i], T1[i]);
    T0[2 * N - 1] = subc(T0[2 * N - 1], T1[2 * N - 1]);
    T0[N] = add_cc(T0[N], P::mod(0));
#pragma unroll
    for (int i = 1; i < N - 1; i++) T0[N + i] = addc_cc(T0[N + i], P::mod(i));
    T0[2 * N - 1] = addc(T0[2 * N - 1], P::mod(N - 1));
#else
    { uint64_t br = 0; for (int i = 0; i < 2 * N; i++) { uint64_t d = (uint64_t)T2[i] - T0[i] - br; T2[i] = (uint32_t)d; br = (d >> 32) & 1; } }
    { uint64_t br = 0; for (int i = 0; i < 2 * N; i++) { uint64_t d = (uint64_t)T2[i] - T1[i] - br; T2[i] = (uint32_t)d; br = (d >> 32) & 1; } }
    { uint64_t br = 0; for (int i = 0; i < 2 * N; i++) { uint64_t d = (uint64_t)T0[i] - T1[i] - br; T0[i] = (uint32_t)d; br = (d >> 32) & 1; } }
    { uint64_t c = 0; for (int i = 0; i < N; i++) { c += (uint64_t)T0[N + i] + P::mod(i); T0[N + i] = (uint32_t)c; c >>= 32; } }
#endif
    Fp2<P> z;
    z.a1 = fp_redc_wide<P, 1>(T2);    // < 2 q^2 < q R / 2: redc_half <= q plus T_hi < q / 2
    z.a0 = fp_redc_wide<P, 2>(T0);    // < q R + q^2:       redc_half <= q plus T_hi < 1.25 q
    return z;
}
#if defined(__CUDA_ARCH__) && defined(GMSM_MUL_NOINLINE)
template <class P>
__device__ __noinline__ Fp2<P> fp2_mul_lazy_ni(Fp2<P> x, Fp2<P> y) {
  return fp2_mul_lazy_inline(x, y);
}
#endif
#endif

// Karatsuba, 3 fp.Mul (e2_bn254.go:28-38; e2_bls377.go:12-23 with the a1*b1 term times 5)
// GMSM_FP2_DOT2 = 1 (experimental): z0 = x0 y0 + x1 (beta y1) and z1 = x0 y1 + x1 y0 as two fused two-product reductions
// (fp_dot2, field.cuh): 4 products + 2 reductions = 400 IMAD.WIDE for N = 8 against Karatsuba's 3 x 136 = 408, without the
// five additions / subtractions Karatsuba pays around its products.  Same unique reduced values.
template <class P>
GMSM_HD Fp2<P> f_mul(const Fp2<P>& x, const Fp2<P>& y) {
  static_assert(P::FP2_NONRES == -1 || P::FP2_NONRES == -5, "supported quadratic non-residues");
#if defined(GMSM_FP2_LAZY)
  if constexpr (P::FP2_NONRES == -1 && (P::mod(P::N - 1) >> 30) == 0) {
#if defined(__CUDA_ARCH__) && defined(GMSM_MUL_NOINLINE)
    return fp2_mul_lazy_ni<P>(x, y);
#else
    return fp2_mul_lazy_inline(x, y);
#endif
  }
#endif
#if defined(GMSM_FP2_DOT2) && defined(GMSM_DOT2)
  Fp2<P> z;
  const Fp<P> by1 = (P::FP2_NONRES == -5) ? fp_neg(fp_mul_by5(y.a1)) : fp_neg(y.a1);
  z.a0 = fp_dot2(x.a0, y.a0, x.a1, by1);
  z.a1 = fp_dot2(x.a0, y.a1, x.a1, y.a0);
  return z;
#else
  Fp<P> a = fp_add(x.a0, x.a1);
  Fp<P> b = fp_add(y.a0, y.a1);
  a = fp_mul(a, b);
  b = fp_mul(x.a0, y.a0);
  Fp<P> c = fp_mul(x.a1, y.a1);
  Fp2<P> z;
  z.a1 = fp_sub(fp_sub(a, b), c);
  if (P::FP2_NONRES == -5) c = fp_mul_by5(c);
  z.a0 = fp_sub(b, c);
  return z;
#endif
}

// 2 fp.Mul (e2_bn254.go:41-51; e2_bls377.go:26-38: (a0+a1)(a0-5a1) + 4 a0 a1)
template <class P>
GMSM_HD Fp2<P> f_sqr(const Fp2<P>& x) {
  Fp<P> a = fp_add(x.a0, x.a1);
  Fp<P> b = (P::FP2_NONRES == -5) ? fp_sub(x.a0, fp_mul_by5(x.a1)) : fp_sub(x.a0, x.a1);
  a = fp_mul(a, b);
  b = fp_dbl(fp_mul(x.a0, x.a1));
  if (P::FP2_NONRES == -5) a = fp_add(a, fp_dbl(b));
  return Fp2<P>{a, b};
}

// x*y + u*v over Fp2.  With GMSM_DOT4 each component is ONE four-product reduction over the base field:
//   z0 = x0 y0 + x1 (beta y1) + u0 v0 + u1 (beta v1),   z1 = x0 y1 + x1 y0 + u0 v1 + u1 v0
// (2 x 328 IMAD.WIDE for N = 8 instead of 4 x 200); otherwise the composition of two products.
template <class P>
GMSM_HD Fp2<P> f_dot2(const Fp2<P>& x, const Fp2<P>& y, const Fp2<P>& u, const Fp2<P>& v) {
#if defined(GMSM_DOT4)
  const Fp<P> by1 = (P::FP2_NONRES == -5) ? fp_neg(fp_mul_by5(y.a1)) : fp_neg(y.a1);
  const Fp<P> bv1 = (P::FP2_NONRES == -5) ? fp_neg(fp_mul_by5(v.a1)) : fp_neg(v.a1);
  Fp2<P> z;
  z.a0 = fp_dot4(x.a0, y.a0, x.a1, by1, u.a0, v.a0, u.a1, bv1);
  z.a1 = fp_dot4(x.a0, y.a1, x.a1, y.a0, u.a0, v.a1, u.a1, v.a0);
  return z;
#else
  return f_add(f_mul(x, y), f_mul(u, v));
#endif
}

// (a0 - a1 u) / (a0^2 + a1^2)   (e2_bn254.go:61-73)
template <class P>
GMSM_HD Fp2<P> f_inv(const Fp2<P>& x) {
  Fp<P> t0 = fp_sqr(x.a0);
  Fp<P> t1 = fp_sqr(x.a1);
  if (P::FP2_NONRES == -5) t1 = fp_mul_by5(t1);   // norm = a0^2 - beta a1^2
  t0 = fp_add(t0, t1);
  t1 = fp_inv(t0);
  return Fp2<P>{fp_mul(x.a0, t1), fp_neg(fp_mul(x.a1, t1))};
}

}  // namespace gmsm

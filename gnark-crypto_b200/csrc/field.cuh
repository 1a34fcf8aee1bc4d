// Montgomery prime-field arithmetic on 32-bit limbs for sm_100a.
//
// Replaces (reference, /root/reference):
//   fp.Mul / Square  : field/asm/element_4w_amd64.s:208-297, element_6w_amd64.s:282-395,
//                      generic CIOS ecc/bn254/fp/element.go:470-591 (final subtract :583-590)
//   fp.Add/Double/Sub/Neg : ecc/bn254/fp/element.go:386-454
//   fr fromMont      : ecc/bn254/fr/element.go:593-642 (via Bits() :855-859)
//
// Representation is byte-identical to the reference's [L]uint64 little-endian Montgomery form
// (value * 2^(64L) mod q, always fully reduced), read as 2L little-endian uint32 limbs.
//
// Device multiplication: row-wise CIOS with two accumulators of 64-bit-aligned (lo,hi) pairs --
// one aligned on even columns, one on odd columns -- so every 32x32+64 multiply-add is one
// IMAD.WIDE.U32.X (ptxas fuses each mad.lo.cc/madc.hi.cc pair) and the per-row shift by one limb
// is free: the accumulators swap roles every row and the one becoming odd-aligned is shifted two
// limbs by reading the MAD addend at index+2.  The low limb never needs a cross-accumulator add: it
// sums to 0 mod 2^32 after the reduction step and its 1-bit carry is injected as the carry-in of
// the next row's first chain.  2*N^2/2 = N^2 IMAD.WIDE per product half, 2*N^2 total
// (N=8: 128, N=12: 288).  Algorithm validated limb-exactly by tools/sim_montmul.py.
#pragma once
#include <cstdint>

#include "field_consts.cuh"
#include "hd.cuh"

namespace gmsm {

#if defined(GMSM_EMULATE_PTX) && !defined(__CUDACC__)
// ---- emulated carry-chain primitives (host test build only): PTX semantics of CC.CF, one flag per thread ----
static thread_local uint32_t emu_cf = 0;
GMSM_D uint32_t emu_add(uint32_t a, uint32_t b, uint32_t cin, bool set) {
  uint64_t s = (uint64_t)a + b + cin;
  if (set) emu_cf = (uint32_t)(s >> 32);
  return (uint32_t)s;
}
GMSM_D uint32_t emu_sub(uint32_t a, uint32_t b, uint32_t bin, bool set) {
  uint64_t d = (uint64_t)a - b - bin;
  if (set) emu_cf = (uint32_t)(d >> 32) & 1;
  return (uint32_t)d;
}
GMSM_D uint32_t add_cc(uint32_t a, uint32_t b) { return emu_add(a, b, 0, true); }
GMSM_D uint32_t addc_cc(uint32_t a, uint32_t b) { return emu_add(a, b, emu_cf, true); }
GMSM_D uint32_t addc(uint32_t a, uint32_t b) { return emu_add(a, b, emu_cf, false); }
GMSM_D uint32_t sub_cc(uint32_t a, uint32_t b) { return emu_sub(a, b, 0, true); }
GMSM_D uint32_t subc_cc(uint32_t a, uint32_t b) { return emu_sub(a, b, emu_cf, true); }
GMSM_D uint32_t subc(uint32_t a, uint32_t b) { return emu_sub(a, b, emu_cf, false); }
GMSM_D uint32_t mad_lo_cc(uint32_t a, uint32_t b, uint32_t c) { return emu_add((uint32_t)((uint64_t)a * b), c, 0, true); }
GMSM_D uint32_t madc_lo_cc(uint32_t a, uint32_t b, uint32_t c) { return emu_add((uint32_t)((uint64_t)a * b), c, emu_cf, true); }
GMSM_D uint32_t madc_hi_cc(uint32_t a, uint32_t b, uint32_t c) { return emu_add((uint32_t)(((uint64_t)a * b) >> 32), c, emu_cf, true); }
GMSM_D uint32_t madc_hi(uint32_t a, uint32_t b, uint32_t c) { return emu_add((uint32_t)(((uint64_t)a * b) >> 32), c, emu_cf, false); }
// a dropped carry-out must be zero: checked in the emulated build, free on the device
#define GMSM_NO_CARRY() do { if (emu_cf) __builtin_trap(); } while (0)
#elif defined(__CUDA_ARCH__)
#define GMSM_NO_CARRY() do { } while (0)
// ---- PTX carry-chain primitives (CC.CF lives across consecutive volatile asm statements) ----
GMSM_D uint32_t add_cc(uint32_t a, uint32_t b) {
  uint32_t r;
  asm volatile("add.cc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}
GMSM_D uint32_t addc_cc(uint32_t a, uint32_t b) {
  uint32_t r;
  asm volatile("addc.cc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}
GMSM_D uint32_t addc(uint32_t a, uint32_t b) {
  uint32_t r;
  asm volatile("addc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}
GMSM_D uint32_t sub_cc(uint32_t a, uint32_t b) {
  uint32_t r;
  asm volatile("sub.cc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}
GMSM_D uint32_t subc_cc(uint32_t a, uint32_t b) {
  uint32_t r;
  asm volatile("subc.cc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}
GMSM_D uint32_t subc(uint32_t a, uint32_t b) {
  uint32_t r;
  asm volatile("subc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}
GMSM_D uint32_t mad_lo_cc(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t r;
  asm volatile("mad.lo.cc.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
  return r;
}
GMSM_D uint32_t madc_lo_cc(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t r;
  asm volatile("madc.lo.cc.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
  return r;
}
GMSM_D uint32_t madc_hi_cc(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t r;
  asm volatile("madc.hi.cc.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
  return r;
}
GMSM_D uint32_t madc_hi(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t r;
  asm volatile("madc.hi.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
  return r;
}
#endif

template <class P>
struct Fp {
  static constexpr int N = P::N;
  using Params = P;
  uint32_t l[N];

  GMSM_HD static Fp zero() {
    Fp r;
#pragma unroll
    for (int i = 0; i < N; i++) r.l[i] = 0;
    return r;
  }
  GMSM_HD static Fp one() {  // R mod q  (SetOne, fp/element.go:194-200)
    Fp r;
#pragma unroll
    for (int i = 0; i < N; i++) r.l[i] = P::one(i);
    return r;
  }
  GMSM_HD bool is_zero() const {  // fp/element.go:221
    uint32_t o = 0;
#pragma unroll
    for (int i = 0; i < N; i++) o |= l[i];
    return o == 0;
  }
  GMSM_HD bool operator==(const Fp& b) const {
    uint32_t o = 0;
#pragma unroll
    for (int i = 0; i < N; i++) o |= l[i] ^ b.l[i];
    return o == 0;
  }
  GMSM_HD bool operator!=(const Fp& b) const { return !(*this == b); }
};

// Modulus limb as a MULTIPLICAND.  Normally the generated constant (an immediate operand of IMAD.WIDE).  A modulus with
// sparse limbs (bls12-377: 0x00000001, 0x8508c000, 0x30000000, ...) tempts ptxas into strength-reducing those products, which
// splits the fused mad.lo.cc / madc.hi.cc pairs into IMAD.HI + IMAD.X -- two multiplier-pipe slots instead of one (measured:
// bls12-377 G1 0.434 ns per mixed addition against bls12-381's 0.377 with identical source).  For such fields
// (Params::MOD_IN_CONST_BANK) the multiplicand is read from __constant__ memory instead: a constant-bank operand costs no
// register and hides the value from the optimiser.  Host builds and additive uses keep the immediate.
template <class P>
GMSM_HD uint32_t invm() {   // -q^-1 mod 2^32 as a multiplicand: see modm (for bls12-377 it is 0xffffffff, i.e. m = -t0)
#if defined(__CUDA_ARCH__)
  if constexpr (P::MOD_IN_CONST_BANK) return P::mod_cb(P::N);
  else
#endif
  return P::INV;
}
template <class P>
GMSM_HD uint32_t modm(int j) {
#if defined(__CUDA_ARCH__)
  if constexpr (P::MOD_IN_CONST_BANK) return P::mod_cb(j);    // (generated next to the constants: a __constant__ array)
  else
#endif
  return P::mod(j);
}

// k * q < 2^(32N), evaluated at compile time from the modulus limbs: the bound the fused multi-product reductions need for
// their intermediate frames (fp_dot4: frames below 5q)
template <class P>
GMSM_HD constexpr bool mod_multiple_fits(uint32_t k) {
  uint64_t c = 0;
  for (int i = 0; i < P::N; i++) c = ((uint64_t)P::mod(i) * k + (c >> 32));
  return (c >> 32) == 0;
}

// r = (a >= q) ? a - q : a, for a value a + carry * 2^(32N) < 2q.  carry is always 0 for the moduli with a spare top bit
// (2q < 2^(32N)); the full-width moduli (secp256k1 fp and fr, P::FULL) hand in the carry-out of the addition / the carry limb of
// the multiplier: a - q then wraps to the right N limbs
template <class P>
GMSM_HD void fp_reduce_once(Fp<P>& a, uint32_t carry = 0) {
  constexpr int N = P::N;
  uint32_t t[N];
#if defined(GMSM_PTX_PATH)
  t[0] = sub_cc(a.l[0], P::mod(0));
#pragma unroll
  for (int i = 1; i < N; i++) t[i] = subc_cc(a.l[i], P::mod(i));
  uint32_t borrow = subc(0, 0);  // 0xffffffff if a < q
  if constexpr (P::FULL) borrow = carry ? 0u : borrow;
#pragma unroll
  for (int i = 0; i < N; i++) a.l[i] = borrow ? a.l[i] : t[i];
#else
  uint64_t br = 0;
  for (int i = 0; i < N; i++) {
    uint64_t d = (uint64_t)a.l[i] - P::mod(i) - br;
    t[i] = (uint32_t)d;
    br = (d >> 32) & 1;
  }
  if (!br || carry)
    for (int i = 0; i < N; i++) a.l[i] = t[i];
#endif
}

// fp.Add  (fp/element.go:386-401): a, b < q
template <class P>
GMSM_HD Fp<P> fp_add(const Fp<P>& a, const Fp<P>& b) {
  constexpr int N = P::N;
  Fp<P> r;
#if defined(GMSM_PTX_PATH)
  uint32_t c = 0;
  r.l[0] = add_cc(a.l[0], b.l[0]);
#pragma unroll
  for (int i = 1; i < N - 1; i++) r.l[i] = addc_cc(a.l[i], b.l[i]);
  if constexpr (P::FULL) {
    r.l[N - 1] = addc_cc(a.l[N - 1], b.l[N - 1]);
    c = addc(0, 0);
  } else {
    r.l[N - 1] = addc(a.l[N - 1], b.l[N - 1]);  // q < 2^(32N-1): no carry out
  }
#else
  uint64_t c = 0;
  for (int i = 0; i < N; i++) {
    c += (uint64_t)a.l[i] + b.l[i];
    r.l[i] = (uint32_t)c;
    c >>= 32;
  }
#endif
  fp_reduce_once(r, (uint32_t)c);
  return r;
}

// fp.Double (fp/element.go:403-418)
template <class P>
GMSM_HD Fp<P> fp_dbl(const Fp<P>& a) {
  return fp_add(a, a);
}

// fp.Sub (fp/element.go:420-438)
template <class P>
GMSM_HD Fp<P> fp_sub(const Fp<P>& a, const Fp<P>& b) {
  constexpr int N = P::N;
  Fp<P> r;
#if defined(GMSM_PTX_PATH)
  r.l[0] = sub_cc(a.l[0], b.l[0]);
#pragma unroll
  for (int i = 1; i < N; i++) r.l[i] = subc_cc(a.l[i], b.l[i]);
  uint32_t mask = subc(0, 0);  // all ones if borrow
  r.l[0] = add_cc(r.l[0], P::mod(0) & mask);
#pragma unroll
  for (int i = 1; i < N - 1; i++) r.l[i] = addc_cc(r.l[i], P::mod(i) & mask);
  r.l[N - 1] = addc(r.l[N - 1], P::mod(N - 1) & mask);
#else
  uint64_t br = 0;
  for (int i = 0; i < N; i++) {
    uint64_t d = (uint64_t)a.l[i] - b.l[i] - br;
    r.l[i] = (uint32_t)d;
    br = (d >> 32) & 1;
  }
  if (br) {
    uint64_t c = 0;
    for (int i = 0; i < N; i++) {
      c += (uint64_t)r.l[i] + P::mod(i);
      r.l[i] = (uint32_t)c;
      c >>= 32;
    }
  }
#endif
  return r;
}

// fp.Neg (fp/element.go:440-454): Neg(0) = 0
template <class P>
GMSM_HD Fp<P> fp_neg(const Fp<P>& a) {
  return fp_sub(Fp<P>::zero(), a);
}

// ------------------------------------------------------------------------------------------
// Montgomery multiplication  z = x*y*R^-1 mod q   (F1)
// ------------------------------------------------------------------------------------------
// Textbook CIOS on 32-bit limbs with the two extra words (_mulGeneric, fp/element.go:470-591, at half the word size): the host
// build's multiplier (the carry limb t[N] joins the final subtraction: zero for the moduli with a spare top bit, live for the
// FULL-width ones) and the reference the device formulation below is tested against.
template <class P>
GMSM_HD Fp<P> fp_mul_cios(const Fp<P>& x, const Fp<P>& y) {
  constexpr int N = P::N;
  Fp<P> r;
  uint32_t t[N + 2];
#pragma unroll
  for (int i = 0; i < N + 2; i++) t[i] = 0;
#pragma unroll
  for (int i = 0; i < N; i++) {
    uint64_t c = 0;
#pragma unroll
    for (int j = 0; j < N; j++) {
      c += (uint64_t)x.l[j] * y.l[i] + t[j];
      t[j] = (uint32_t)c;
      c >>= 32;
    }
    c += t[N];
    t[N] = (uint32_t)c;
    t[N + 1] = (uint32_t)(c >> 32);
    uint32_t m = t[0] * P::INV;
    c = (uint64_t)m * P::mod(0) + t[0];
    c >>= 32;
#pragma unroll
    for (int j = 1; j < N; j++) {
      c += (uint64_t)m * P::mod(j) + t[j];
      t[j - 1] = (uint32_t)c;
      c >>= 32;
    }
    c += t[N];
    t[N - 1] = (uint32_t)c;
    t[N] = t[N + 1] + (uint32_t)(c >> 32);
  }
#pragma unroll
  for (int i = 0; i < N; i++) r.l[i] = t[i];
  fp_reduce_once(r, t[N]);
  return r;
}

template <class P>
GMSM_HD Fp<P> fp_mul_inline(const Fp<P>& x, const Fp<P>& y) {
  constexpr int N = P::N;
  Fp<P> r;
#if defined(GMSM_PTX_PATH) && !defined(GMSM_PORTABLE_MUL)
  // Two accumulators, N+2 slots each: [0..N-1] limbs, [N] carry limb, [N+1] always zero.
  // Full-width moduli (P::FULL, secp256k1): T < 2q no longer fits N limbs, so the two carries that the spare top bit makes
  // zero are kept -- the carry out of the odd accumulator's reduction chain (step 5) goes to ITS carry limb, which the next
  // row (where that accumulator is the even one) adds to instead of overwriting, and the last row's joins the final sum as
  // limb N, the carry fp_reduce_once takes.  Two more ADDCs per row; everything else is unchanged.
  uint32_t A[N + 2], B[N + 2];
#pragma unroll
  for (int i = 0; i < N + 2; i++) A[i] = B[i] = 0;
  uint32_t dprev = 0;  // dangling limb of the previous row (column 0 of the current frame)
  uint32_t e0prev = 0; // low limb of the previous row's Ev after reduction (e0prev + dprev == 0 mod 2^32)
#pragma unroll
  for (int i = 0; i < N; i++) {
    uint32_t* Ev = (i & 1) ? B : A;
    uint32_t* Od = (i & 1) ? A : B;
    const uint32_t bi = y.l[i];
    // frame shift from the previous row: the previous Ev is this row's pending Od:
    //   k  = carry(e0prev + dprev)  -> carry-in of this row's first chain
    //   d  = prevEv[1] = Od[1]      -> this row's dangling limb (column 0)
    const uint32_t d = (i == 0) ? 0u : Od[1];
    // step 1: Ev += x_even * bi
    if (i == 0) {
      Ev[0] = mad_lo_cc(x.l[0], bi, Ev[0]);
    } else {
      (void)add_cc(e0prev, dprev);
      Ev[0] = madc_lo_cc(x.l[0], bi, Ev[0]);
    }
    Ev[1] = madc_hi_cc(x.l[0], bi, Ev[1]);
#pragma unroll
    for (int j = 2; j < N; j += 2) {
      Ev[j] = madc_lo_cc(x.l[j], bi, Ev[j]);
      Ev[j + 1] = madc_hi_cc(x.l[j], bi, Ev[j + 1]);
    }
    if constexpr (P::FULL) Ev[N] = addc(Ev[N], 0);   // (Ev was the previous row's Od: its carry limb is live)
    else Ev[N] = addc(0, 0);
    // step 2: Od = (Od >> 2 limbs) + x_odd * bi   (no carry out; Od[N+1] == 0)
    Od[0] = mad_lo_cc(x.l[1], bi, Od[2]);
    Od[1] = madc_hi_cc(x.l[1], bi, Od[3]);
#pragma unroll
    for (int j = 2; j < N; j += 2) {
      Od[j] = madc_lo_cc(x.l[j + 1], bi, Od[j + 2]);
      Od[j + 1] = madc_hi_cc(x.l[j + 1], bi, Od[j + 3]);
    }
    Od[N] = 0;  // stale carry limb consumed by the shift
    // step 3
    const uint32_t m = (Ev[0] + d) * invm<P>();
    // step 4: Ev += q_even * m
    Ev[0] = mad_lo_cc(modm<P>(0), m, Ev[0]);
    Ev[1] = madc_hi_cc(modm<P>(0), m, Ev[1]);
#pragma unroll
    for (int j = 2; j < N; j += 2) {
      Ev[j] = madc_lo_cc(modm<P>(j), m, Ev[j]);
      Ev[j + 1] = madc_hi_cc(modm<P>(j), m, Ev[j + 1]);
    }
    Ev[N] = addc(Ev[N], 0);
    // step 5: Od += q_odd * m  (no carry out)
    Od[0] = mad_lo_cc(modm<P>(1), m, Od[0]);
    Od[1] = madc_hi_cc(modm<P>(1), m, Od[1]);
#pragma unroll
    for (int j = 2; j < N; j += 2) {
      Od[j] = madc_lo_cc(modm<P>(j + 1), m, Od[j]);
      Od[j + 1] = madc_hi_cc(modm<P>(j + 1), m, Od[j + 1]);
    }
    if constexpr (P::FULL) Od[N] = addc(0, 0);
    e0prev = Ev[0];
    dprev = d;
  }
  // After the last row (N even): last Ev = B, last Od = A.
  //   result = A[0..N-1] + B[1] + carry(B[0] + dprev) + 2^32 * B[2..N]
  (void)add_cc(e0prev, dprev);
  r.l[0] = addc_cc(A[0], B[1]);
#pragma unroll
  for (int i = 1; i < N - 1; i++) r.l[i] = addc_cc(A[i], B[i + 1]);
  if constexpr (P::FULL) {
    r.l[N - 1] = addc_cc(A[N - 1], B[N]);
    fp_reduce_once(r, addc(A[N], 0));
  } else {
    r.l[N - 1] = addc(A[N - 1], B[N]);
    fp_reduce_once(r);
  }
#else
  return fp_mul_cios(x, y);
#endif
  return r;
}

// Out-of-line copy of the multiplier (operands and result travel in registers under the device ABI).
// One mixed add inlines 10 (G1) .. 28 (G2) multiplications of ~220 (N=8) / ~480 (N=12) SASS instructions:
// 35 .. 100+ KB of straight-line code against a 32 KB L1.5 instruction cache.  GMSM_MUL_NOINLINE trades a
// CALL/RET pair per multiplication for an instruction footprint that fits.
#if defined(__CUDA_ARCH__) && defined(GMSM_MUL_NOINLINE)
template <class P> GMSM_HD Fp<P> fp_mul_karatsuba(const Fp<P>& x, const Fp<P>& y);
template <class P>
__device__ __noinline__ Fp<P> fp_mul_ni(Fp<P> x, Fp<P> y) {
#if defined(GMSM_MUL_KARATSUBA)
  if constexpr (P::N % 4 == 0 && (P::mod(P::N - 1) >> 30) == 0) return fp_mul_karatsuba(x, y);
  else
#endif
  return fp_mul_inline(x, y);
}
template <class P>
GMSM_HD Fp<P> fp_mul(const Fp<P>& x, const Fp<P>& y) {
  return fp_mul_ni<P>(x, y);
}
#else
template <class P> GMSM_HD Fp<P> fp_mul_karatsuba(const Fp<P>& x, const Fp<P>& y);   // (defined with the separated routines below)
template <class P>
GMSM_HD Fp<P> fp_mul(const Fp<P>& x, const Fp<P>& y) {
#if defined(GMSM_MUL_KARATSUBA)
  if constexpr (P::N % 4 == 0 && (P::mod(P::N - 1) >> 30) == 0) return fp_mul_karatsuba(x, y);
  else
#endif
  return fp_mul_inline(x, y);
}
#endif

// Dedicated Montgomery squaring (experimental: -DGMSM_SQR_DEDICATED=1, default off -- the reference's amd64 Square also
// just calls mul(x, x), fp/element_amd64.go:51-55).  Same row-wise CIOS with the even / odd accumulator pair as
// fp_mul_inline, but row i only multiplies x_i by the limbs j >= i of the operand: x_i itself on the diagonal and
// twice the limbs above it (2 * (x >> 32(i+1)): the limbs of 2x, except that limb i+1 takes no bit from x_i) -- the
// doubling cannot overflow the N limbs because the supported moduli leave at least two spare top bits -- so
// N(N-1)/2 of the N^2 product IMAD.WIDEs disappear (28 of 64 for N = 8; the N^2 + N of the reduction stay: 108 instead of
// 136 per squaring).  Skipped even columns still ripple the row's 1-bit carry-in (ADDC on the ALU pipe, which has
// headroom: DESIGN.md section 5); skipped odd columns are plain moves of the frame shift.  The total added over the
// rows is exactly x^2, so the result and its < 2q bound are unchanged; intermediate frames stay below 3q < 2^(32N).
// The dropped-carry assertions (GMSM_NO_CARRY) are checked by the emulated host build like those of the multiplier.
#if defined(GMSM_SQR_DEDICATED) && defined(GMSM_PTX_PATH) && !defined(GMSM_PORTABLE_MUL)
template <class P>
GMSM_HD Fp<P> fp_sqr_inline(const Fp<P>& x) {
  constexpr int N = P::N;
  static_assert((P::mod(N - 1) >> 30) == 0, "needs two spare top bits (2x in N limbs, frames below 3q)");
  Fp<P> r;
  uint32_t x2[N];   // limbs of 2x
  x2[0] = x.l[0] << 1;
#pragma unroll
  for (int j = 1; j < N; j++) x2[j] = (x.l[j] << 1) | (x.l[j - 1] >> 31);
  uint32_t A[N + 2], B[N + 2];
#pragma unroll
  for (int i = 0; i < N + 2; i++) A[i] = B[i] = 0;
  uint32_t dprev = 0, e0prev = 0;
#pragma unroll
  for (int i = 0; i < N; i++) {
    uint32_t* Ev = (i & 1) ? B : A;
    uint32_t* Od = (i & 1) ? A : B;
    const uint32_t bi = x.l[i];
    const uint32_t d = (i == 0) ? 0u : Od[1];
    // step 1: Ev += (operand limbs at even j >= i) * bi; columns below i only carry the row's carry-in upwards
    if (i != 0) (void)add_cc(e0prev, dprev);
    bool chain = (i != 0);   // is a carry chain running?  (compile-time after unrolling)
#pragma unroll
    for (int j = 0; j < N; j += 2) {
      if (j < i) {
        Ev[j] = addc_cc(Ev[j], 0);
        Ev[j + 1] = addc_cc(Ev[j + 1], 0);
      } else {
        const uint32_t xj = (j == i) ? x.l[j] : (j == i + 1) ? (x.l[j] << 1) : x2[j];   // 2 * (the limbs above i): no bit from x_i
        Ev[j] = chain ? madc_lo_cc(xj, bi, Ev[j]) : mad_lo_cc(xj, bi, Ev[j]);
        Ev[j + 1] = madc_hi_cc(xj, bi, Ev[j + 1]);
      }
      chain = true;
    }
    Ev[N] = addc(0, 0);
    // step 2: Od = (Od >> 2 limbs) + (operand limbs at odd j >= i) * bi   (no carry out; Od[N+1] == 0)
    chain = false;
#pragma unroll
    for (int j = 0; j < N; j += 2) {
      if (j + 1 < i) {
        Od[j] = Od[j + 2];
        Od[j + 1] = Od[j + 3];
      } else {
        const uint32_t xj = (j + 1 == i) ? x.l[j + 1] : (j == i) ? (x.l[j + 1] << 1) : x2[j + 1];
        Od[j] = chain ? madc_lo_cc(xj, bi, Od[j + 2]) : mad_lo_cc(xj, bi, Od[j + 2]);
        Od[j + 1] = madc_hi_cc(xj, bi, Od[j + 3]);
        chain = true;
      }
    }
    if (chain) GMSM_NO_CARRY();
    Od[N] = 0;
    // steps 3-5: the reduction of fp_mul_inline, unchanged
    const uint32_t m = (Ev[0] + d) * invm<P>();
    Ev[0] = mad_lo_cc(modm<P>(0), m, Ev[0]);
    Ev[1] = madc_hi_cc(modm<P>(0), m, Ev[1]);
#pragma unroll
    for (int j = 2; j < N; j += 2) {
      Ev[j] = madc_lo_cc(modm<P>(j), m, Ev[j]);
      Ev[j + 1] = madc_hi_cc(modm<P>(j), m, Ev[j + 1]);
    }
    Ev[N] = addc(Ev[N], 0);
    Od[0] = mad_lo_cc(modm<P>(1), m, Od[0]);
    Od[1] = madc_hi_cc(modm<P>(1), m, Od[1]);
#pragma unroll
    for (int j = 2; j < N; j += 2) {
      Od[j] = madc_lo_cc(modm<P>(j + 1), m, Od[j]);
      Od[j + 1] = madc_hi_cc(modm<P>(j + 1), m, Od[j + 1]);
    }
    GMSM_NO_CARRY();
    e0prev = Ev[0];
    dprev = d;
  }
  (void)add_cc(e0prev, dprev);
  r.l[0] = addc_cc(A[0], B[1]);
#pragma unroll
  for (int i = 1; i < N - 1; i++) r.l[i] = addc_cc(A[i], B[i + 1]);
  r.l[N - 1] = addc(A[N - 1], B[N]);
  fp_reduce_once(r);
  return r;
}
#if defined(__CUDA_ARCH__) && defined(GMSM_MUL_NOINLINE)
template <class P>
__device__ __noinline__ Fp<P> fp_sqr_ni(Fp<P> x) {
  return fp_sqr_inline(x);
}
template <class P>
GMSM_HD Fp<P> fp_sqr(const Fp<P>& x) {
  if constexpr ((P::mod(P::N - 1) >> 30) == 0) return fp_sqr_ni<P>(x);
  else return fp_mul(x, x);   // one spare bit only (bls12-381 fr): keep the multiplier
}
#else
template <class P>
GMSM_HD Fp<P> fp_sqr(const Fp<P>& x) {
  if constexpr ((P::mod(P::N - 1) >> 30) == 0) return fp_sqr_inline(x);
  else return fp_mul(x, x);
}
#endif
#else
template <class P>
GMSM_HD Fp<P> fp_sqr(const Fp<P>& x) {
  return fp_mul(x, x);
}
#endif

// Sum of two products with ONE reduction (experimental: -DGMSM_DOT2=1, default off):  z = (x*y + u*v) * R^-1 mod q.
// The rows of the CIOS take both products (two MAD chains per accumulator and row) and share the reduction steps:
// 2 N^2 product + N^2 + N reduction IMAD.WIDEs = 200 for N = 8 instead of 272 for two multiplications, and one
// conditional subtraction instead of two plus the fp_sub -- no extra ALU work at all.  Used for the y-coordinate of the
// point additions (Y3 = (Q - X3) * R + (-Y1) * PPP, curve.cuh), 5 % of a mixed addition's multiplier work.  Needs the
// two spare top bits like the dedicated squaring: frames stay below 3q < 2^(32N), the result below (2q/2^(32N) + 1) q < 2q.
#if defined(GMSM_DOT2) && defined(GMSM_PTX_PATH) && !defined(GMSM_PORTABLE_MUL)
template <class P>
GMSM_HD Fp<P> fp_dot2_inline(const Fp<P>& x, const Fp<P>& y, const Fp<P>& u, const Fp<P>& v) {
  constexpr int N = P::N;
  static_assert((P::mod(N - 1) >> 30) == 0, "needs two spare top bits (frames below 3q)");
  Fp<P> r;
  uint32_t A[N + 2], B[N + 2];
#pragma unroll
  for (int i = 0; i < N + 2; i++) A[i] = B[i] = 0;
  uint32_t dprev = 0, e0prev = 0;
#pragma unroll
  for (int i = 0; i < N; i++) {
    uint32_t* Ev = (i & 1) ? B : A;
    uint32_t* Od = (i & 1) ? A : B;
    const uint32_t bi = y.l[i], vi = v.l[i];
    const uint32_t d = (i == 0) ? 0u : Od[1];
    // step 1a: Ev += x_even * bi (with the row's carry-in), 1b: Ev += u_even * vi
    if (i == 0) {
      Ev[0] = mad_lo_cc(x.l[0], bi, Ev[0]);
    } else {
      (void)add_cc(e0prev, dprev);
      Ev[0] = madc_lo_cc(x.l[0], bi, Ev[0]);
    }
    Ev[1] = madc_hi_cc(x.l[0], bi, Ev[1]);
#pragma unroll
    for (int j = 2; j < N; j += 2) {
      Ev[j] = madc_lo_cc(x.l[j], bi, Ev[j]);
      Ev[j + 1] = madc_hi_cc(x.l[j], bi, Ev[j + 1]);
    }
    Ev[N] = addc(0, 0);
    Ev[0] = mad_lo_cc(u.l[0], vi, Ev[0]);
    Ev[1] = madc_hi_cc(u.l[0], vi, Ev[1]);
#pragma unroll
    for (int j = 2; j < N; j += 2) {
      Ev[j] = madc_lo_cc(u.l[j], vi, Ev[j]);
      Ev[j + 1] = madc_hi_cc(u.l[j], vi, Ev[j + 1]);
    }
    Ev[N] = addc(Ev[N], 0);
    // step 2a: Od = (Od >> 2 limbs) + x_odd * bi, 2b: Od += u_odd * vi   (no carry out of either)
    Od[0] = mad_lo_cc(x.l[1], bi, Od[2]);
    Od[1] = madc_hi_cc(x.l[1], bi, Od[3]);
#pragma unroll
    for (int j = 2; j < N; j += 2) {
      Od[j] = madc_lo_cc(x.l[j + 1], bi, Od[j + 2]);
      Od[j + 1] = madc_hi_cc(x.l[j + 1], bi, Od[j + 3]);
    }
    GMSM_NO_CARRY();
    Od[N] = 0;
    Od[0] = mad_lo_cc(u.l[1], vi, Od[0]);
    Od[1] = madc_hi_cc(u.l[1], vi, Od[1]);
#pragma unroll
    for (int j = 2; j < N; j += 2) {
      Od[j] = madc_lo_cc(u.l[j + 1], vi, Od[j]);
      Od[j + 1] = madc_hi_cc(u.l[j + 1], vi, Od[j + 1]);
    }
    GMSM_NO_CARRY();
    // steps 3-5: the reduction of fp_mul_inline, unchanged
    const uint32_t m = (Ev[0] + d) * invm<P>();
    Ev[0] = mad_lo_cc(modm<P>(0), m, Ev[0]);
    Ev[1] = madc_hi_cc(modm<P>(0), m, Ev[1]);
#pragma unroll
    for (int j = 2; j < N; j += 2) {
      Ev[j] = madc_lo_cc(modm<P>(j), m, Ev[j]);
      Ev[j + 1] = madc_hi_cc(modm<P>(j), m, Ev[j + 1]);
    }
    Ev[N] = addc(Ev[N], 0);
    Od[0] = mad_lo_cc(modm<P>(1), m, Od[0]);
    Od[1] = madc_hi_cc(modm<P>(1), m, Od[1]);
#pragma unroll
    for (int j = 2; j < N; j += 2) {
      Od[j] = madc_lo_cc(modm<P>(j + 1), m, Od[j]);
      Od[j + 1] = madc_hi_cc(modm<P>(j + 1), m, Od[j + 1]);
    }
    GMSM_NO_CARRY();
    e0prev = Ev[0];
    dprev = d;
  }
  (void)add_cc(e0prev, dprev);
  r.l[0] = addc_cc(A[0], B[1]);
#pragma unroll
  for (int i = 1; i < N - 1; i++) r.l[i] = addc_cc(A[i], B[i + 1]);
  r.l[N - 1] = addc(A[N - 1], B[N]);
  fp_reduce_once(r);
  return r;
}
#if defined(__CUDA_ARCH__) && defined(GMSM_MUL_NOINLINE)
template <class P>
__device__ __noinline__ Fp<P> fp_dot2_ni(Fp<P> x, Fp<P> y, Fp<P> u, Fp<P> v) {
  return fp_dot2_inline(x, y, u, v);
}
#endif
#endif
// Sum of FOUR products with one reduction (GMSM_DOT4, used for the y-coordinate over Fp2: each component of
// (Q - X3) R - Y1 PPP is four base-field products): z = (x0 y0 + x1 y1 + x2 y2 + x3 y3) R^-1 mod q.  4 N^2 + N^2 + N = 328
// IMAD.WIDE for N = 8 instead of 2 x 200 for two fused pairs.  Frames stay below 5q, which must fit the limbs
// (bn254: 5q = 0.945 * 2^256); the result is below (4 q / 2^(32N) + 1) q < 2q.
#if defined(GMSM_DOT4) && defined(GMSM_PTX_PATH) && !defined(GMSM_PORTABLE_MUL)
template <class P>
GMSM_HD Fp<P> fp_dot4_inline(const Fp<P>& x0, const Fp<P>& y0, const Fp<P>& x1, const Fp<P>& y1, const Fp<P>& x2, const Fp<P>& y2,
                             const Fp<P>& x3, const Fp<P>& y3) {
  constexpr int N = P::N;
  static_assert(mod_multiple_fits<P>(5), "needs 5q < 2^(32N) (frames below 5q)");
  Fp<P> r;
  uint32_t A[N + 2], B[N + 2];
#pragma unroll
  for (int i = 0; i < N + 2; i++) A[i] = B[i] = 0;
  uint32_t dprev = 0, e0prev = 0;
  const Fp<P>* xs[4] = {&x0, &x1, &x2, &x3};
  const Fp<P>* ys[4] = {&y0, &y1, &y2, &y3};
#pragma unroll
  for (int i = 0; i < N; i++) {
    uint32_t* Ev = (i & 1) ? B : A;
    uint32_t* Od = (i & 1) ? A : B;
    const uint32_t d = (i == 0) ? 0u : Od[1];
    // step 1: Ev += sum_k x_k,even * y_k[i]  (the row's carry-in rides the first chain)
#pragma unroll
    for (int k = 0; k < 4; k++) {
      const uint32_t bi = ys[k]->l[i];
      const Fp<P>& x = *xs[k];
      if (k == 0 && i != 0) {
        (void)add_cc(e0prev, dprev);
        Ev[0] = madc_lo_cc(x.l[0], bi, Ev[0]);
      } else {
        Ev[0] = mad_lo_cc(x.l[0], bi, Ev[0]);
      }
      Ev[1] = madc_hi_cc(x.l[0], bi, Ev[1]);
#pragma unroll
      for (int j = 2; j < N; j += 2) {
        Ev[j] = madc_lo_cc(x.l[j], bi, Ev[j]);
        Ev[j + 1] = madc_hi_cc(x.l[j], bi, Ev[j + 1]);
      }
      if (k == 0) Ev[N] = addc(0, 0); else Ev[N] = addc(Ev[N], 0);
    }
    // step 2: Od = (Od >> 2 limbs) + sum_k x_k,odd * y_k[i]   (no carry out of any chain)
#pragma unroll
    for (int k = 0; k < 4; k++) {
      const uint32_t bi = ys[k]->l[i];
      const Fp<P>& x = *xs[k];
      if (k == 0) {
        Od[0] = mad_lo_cc(x.l[1], bi, Od[2]);
        Od[1] = madc_hi_cc(x.l[1], bi, Od[3]);
#pragma unroll
        for (int j = 2; j < N; j += 2) {
          Od[j] = madc_lo_cc(x.l[j + 1], bi, Od[j + 2]);
          Od[j + 1] = madc_hi_cc(x.l[j + 1], bi, Od[j + 3]);
        }
        GMSM_NO_CARRY();
        Od[N] = 0;
      } else {
        Od[0] = mad_lo_cc(x.l[1], bi, Od[0]);
        Od[1] = madc_hi_cc(x.l[1], bi, Od[1]);
#pragma unroll
        for (int j = 2; j < N; j += 2) {
          Od[j] = madc_lo_cc(x.l[j + 1], bi, Od[j]);
          Od[j + 1] = madc_hi_cc(x.l[j + 1], bi, Od[j + 1]);
        }
        GMSM_NO_CARRY();
      }
    }
    // steps 3-5: the reduction of fp_mul_inline, unchanged
    const uint32_t m = (Ev[0] + d) * invm<P>();
    Ev[0] = mad_lo_cc(modm<P>(0), m, Ev[0]);
    Ev[1] = madc_hi_cc(modm<P>(0), m, Ev[1]);
#pragma unroll
    for (int j = 2; j < N; j += 2) {
      Ev[j] = madc_lo_cc(modm<P>(j), m, Ev[j]);
      Ev[j + 1] = madc_hi_cc(modm<P>(j), m, Ev[j + 1]);
    }
    Ev[N] = addc(Ev[N], 0);
    Od[0] = mad_lo_cc(modm<P>(1), m, Od[0]);
    Od[1] = madc_hi_cc(modm<P>(1), m, Od[1]);
#pragma unroll
    for (int j = 2; j < N; j += 2) {
      Od[j] = madc_lo_cc(modm<P>(j + 1), m, Od[j]);
      Od[j + 1] = madc_hi_cc(modm<P>(j + 1), m, Od[j + 1]);
    }
    GMSM_NO_CARRY();
    e0prev = Ev[0];
    dprev = d;
  }
  (void)add_cc(e0prev, dprev);
  r.l[0] = addc_cc(A[0], B[1]);
#pragma unroll
  for (int i = 1; i < N - 1; i++) r.l[i] = addc_cc(A[i], B[i + 1]);
  r.l[N - 1] = addc(A[N - 1], B[N]);
  fp_reduce_once(r);
  return r;
}
#if defined(__CUDA_ARCH__) && defined(GMSM_MUL_NOINLINE)
template <class P>
__device__ __noinline__ Fp<P> fp_dot4_ni(Fp<P> x0, Fp<P> y0, Fp<P> x1, Fp<P> y1, Fp<P> x2, Fp<P> y2, Fp<P> x3, Fp<P> y3) {
  return fp_dot4_inline(x0, y0, x1, y1, x2, y2, x3, y3);
}
#endif
#endif
template <class P>
GMSM_HD Fp<P> fp_dot4(const Fp<P>& x0, const Fp<P>& y0, const Fp<P>& x1, const Fp<P>& y1, const Fp<P>& x2, const Fp<P>& y2,
                      const Fp<P>& x3, const Fp<P>& y3);

// x*y + u*v: the fused form above where it is compiled in and the modulus has the spare bits, two products otherwise
template <class P>
GMSM_HD Fp<P> fp_dot2(const Fp<P>& x, const Fp<P>& y, const Fp<P>& u, const Fp<P>& v) {
#if defined(GMSM_DOT2) && defined(GMSM_PTX_PATH) && !defined(GMSM_PORTABLE_MUL)
  if constexpr ((P::mod(P::N - 1) >> 30) == 0) {
#if defined(__CUDA_ARCH__) && defined(GMSM_MUL_NOINLINE)
    return fp_dot2_ni<P>(x, y, u, v);
#else
    return fp_dot2_inline(x, y, u, v);
#endif
  } else
#endif
  {
    return fp_add(fp_mul(x, y), fp_mul(u, v));
  }
}
template <class P>
GMSM_HD Fp<P> fp_dot4(const Fp<P>& x0, const Fp<P>& y0, const Fp<P>& x1, const Fp<P>& y1, const Fp<P>& x2, const Fp<P>& y2,
                      const Fp<P>& x3, const Fp<P>& y3) {
#if defined(GMSM_DOT4) && defined(GMSM_PTX_PATH) && !defined(GMSM_PORTABLE_MUL)
  if constexpr (mod_multiple_fits<P>(5)) {   // bn254: 5q = 0.945 * 2^256; a q in [0.2, 0.25) * 2^(32N) takes two fp_dot2
#if defined(__CUDA_ARCH__) && defined(GMSM_MUL_NOINLINE)
    return fp_dot4_ni<P>(x0, y0, x1, y1, x2, y2, x3, y3);
#else
    return fp_dot4_inline(x0, y0, x1, y1, x2, y2, x3, y3);
#endif
  } else
#endif
  {
    return fp_add(fp_dot2(x0, y0, x1, y1), fp_dot2(x2, y2, x3, y3));
  }
}

// ------------------------------------------------------------------------------------------
// Separated product / reduction (experimental building blocks: -DGMSM_FP2_LAZY=1 uses them for the Fp2 product)
//   fp_mul_wide : t[0..2N) = x * y, plain 2N-limb product (operands are any N-limb integers)
//   fp_redc_wide: T * R^-1 mod q for a 2N-limb T < ~3 q R  =  redc_half(T_lo) + T_hi, where redc_half(v) = (v + m q) / R is the
//                 reduction half of the CIOS above (fp_mul_inline with y = 1: same frames, same carry injection, the product
//                 MADs dropped: N^2 + N IMAD.WIDE)
// Same IMAD.WIDE count as the interleaved CIOS (N^2 + N^2 + N), but sums / differences of several double-width products can
// share ONE reduction (lazy reduction: the Fp2 product of e2_bn254.go:28-38 needs 3 products and 2 reductions, 336 instead of
// 3 x 136 = 408 IMAD.WIDE for N = 8).
// ------------------------------------------------------------------------------------------
template <int N>
GMSM_HD void mul_wide_limbs(const uint32_t* x, const uint32_t* y, uint32_t* t) {
  static_assert(N % 2 == 0, "even limb count");
#if defined(GMSM_PTX_PATH) && !defined(GMSM_PORTABLE_MUL)
  // two accumulators of 64-bit-aligned (lo, hi) pairs: E holds the pairs at even limb positions, O at odd ones; the product
  // x_j * y_i sits at position i + j.  Every chain covers N contiguous limbs and drops its carry into the next, still small, limb.
  uint32_t E[2 * N + 2], O[2 * N + 2];
#pragma unroll
  for (int i = 0; i < 2 * N + 2; i++) E[i] = O[i] = 0;
#pragma unroll
  for (int i = 0; i < N; i++) {
    uint32_t* Pe = (i & 1) ? O : E;   // x_even * y_i: positions of the parity of i
    uint32_t* Po = (i & 1) ? E : O;   // x_odd  * y_i: the other parity
    const uint32_t bi = y[i];
    Pe[i] = mad_lo_cc(x[0], bi, Pe[i]);
    Pe[i + 1] = madc_hi_cc(x[0], bi, Pe[i + 1]);
#pragma unroll
    for (int j = 2; j < N; j += 2) {
      Pe[i + j] = madc_lo_cc(x[j], bi, Pe[i + j]);
      Pe[i + j + 1] = madc_hi_cc(x[j], bi, Pe[i + j + 1]);
    }
    Pe[i + N] = addc(Pe[i + N], 0);
    Po[i + 1] = mad_lo_cc(x[1], bi, Po[i + 1]);
    Po[i + 2] = madc_hi_cc(x[1], bi, Po[i + 2]);
#pragma unroll
    for (int j = 3; j < N; j += 2) {
      Po[i + j] = madc_lo_cc(x[j], bi, Po[i + j]);
      Po[i + j + 1] = madc_hi_cc(x[j], bi, Po[i + j + 1]);
    }
    Po[i + N + 1] = addc(Po[i + N + 1], 0);
  }
  t[0] = add_cc(E[0], O[0]);
#pragma unroll
  for (int i = 1; i < 2 * N - 1; i++) t[i] = addc_cc(E[i], O[i]);
  t[2 * N - 1] = addc(E[2 * N - 1], O[2 * N - 1]);
#else
  for (int i = 0; i < 2 * N; i++) t[i] = 0;
  for (int i = 0; i < N; i++) {
    uint64_t c = 0;
    for (int j = 0; j < N; j++) {
      c += (uint64_t)x[j] * y[i] + t[i + j];
      t[i + j] = (uint32_t)c;
      c >>= 32;
    }
    t[i + N] = (uint32_t)c;
  }
#endif
}

template <class P>
GMSM_HD void fp_mul_wide(const uint32_t* x, const uint32_t* y, uint32_t* t) {
  mul_wide_limbs<P::N>(x, y, t);
}

// One level of Karatsuba on top of the plain product (N = 2H, H even): x = xl + xh B, y = yl + yh B with B = 2^(32H),
//   x y = z0 + (zm - z0 - z2) B + z2 B^2,  z0 = xl yl, z2 = xh yh, zm = (xl + xh)(yl + yh)
// three H x H products (3 H^2 = 48 IMAD.WIDE for N = 8 instead of 64) for ~60 more additions; the carry bits of the two
// half sums are handled with masked additions.
template <int N>
GMSM_HD void mul_wide_karatsuba(const uint32_t* x, const uint32_t* y, uint32_t* t) {
  constexpr int H = N / 2;
  static_assert(H % 2 == 0, "N must be a multiple of 4");
  uint32_t sx[H], sy[H], zm[2 * H + 1];
  uint32_t cx, cy;
#if defined(GMSM_PTX_PATH)
  sx[0] = add_cc(x[0], x[H]);
#pragma unroll
  for (int i = 1; i < H; i++) sx[i] = addc_cc(x[i], x[H + i]);
  cx = addc(0, 0);
  sy[0] = add_cc(y[0], y[H]);
#pragma unroll
  for (int i = 1; i < H; i++) sy[i] = addc_cc(y[i], y[H + i]);
  cy = addc(0, 0);
#else
  { uint64_t c = 0; for (int i = 0; i < H; i++) { c += (uint64_t)x[i] + x[H + i]; sx[i] = (uint32_t)c; c >>= 32; } cx = (uint32_t)c; }
  { uint64_t c = 0; for (int i = 0; i < H; i++) { c += (uint64_t)y[i] + y[H + i]; sy[i] = (uint32_t)c; c >>= 32; } cy = (uint32_t)c; }
#endif
  mul_wide_limbs<H>(x, y, t);                  // z0 -> t[0 .. 2H)
  mul_wide_limbs<H>(x + H, y + H, t + 2 * H);  // z2 -> t[2H .. 4H)
  mul_wide_limbs<H>(sx, sy, zm);
  zm[2 * H] = cx & cy;
  const uint32_t mx = 0u - cx, my = 0u - cy;   // all ones if the half sum carried
#if defined(GMSM_PTX_PATH)
  // zm += (cx ? sy : 0) B + (cy ? sx : 0) B      (into limbs H .. 2H, carries into zm[2H])
  zm[H] = add_cc(zm[H], sy[0] & mx);
#pragma unroll
  for (int i = 1; i < H; i++) zm[H + i] = addc_cc(zm[H + i], sy[i] & mx);
  zm[2 * H] = addc(zm[2 * H], 0);
  zm[H] = add_cc(zm[H], sx[0] & my);
#pragma unroll
  for (int i = 1; i < H; i++) zm[H + i] = addc_cc(zm[H + i], sx[i] & my);
  zm[2 * H] = addc(zm[2 * H], 0);
  // zm -= z0; zm -= z2    (the middle term is non-negative: no borrow out of limb 2H)
  zm[0] = sub_cc(zm[0], t[0]);
#pragma unroll
  for (int i = 1; i < 2 * H; i++) zm[i] = subc_cc(zm[i], t[i]);
  zm[2 * H] = subc(zm[2 * H], 0);
  zm[0] = sub_cc(zm[0], t[2 * H]);
#pragma unroll
  for (int i = 1; i < 2 * H; i++) zm[i] = subc_cc(zm[i], t[2 * H + i]);
  zm[2 * H] = subc(zm[2 * H], 0);
  // t += zm B
  t[H] = add_cc(t[H], zm[0]);
#pragma unroll
  for (int i = 1; i <= 2 * H; i++) t[H + i] = addc_cc(t[H + i], zm[i]);
#pragma unroll
  for (int i = 3 * H + 1; i < 4 * H - 1; i++) t[i] = addc_cc(t[i], 0);
  t[4 * H - 1] = addc(t[4 * H - 1], 0);
#else
  { uint64_t c = 0; for (int i = 0; i < H; i++) { c += (uint64_t)zm[H + i] + (sy[i] & mx); zm[H + i] = (uint32_t)c; c >>= 32; } zm[2 * H] += (uint32_t)c; }
  { uint64_t c = 0; for (int i = 0; i < H; i++) { c += (uint64_t)zm[H + i] + (sx[i] & my); zm[H + i] = (uint32_t)c; c >>= 32; } zm[2 * H] += (uint32_t)c; }
  { uint64_t br = 0; for (int i = 0; i < 2 * H; i++) { uint64_t d = (uint64_t)zm[i] - t[i] - br; zm[i] = (uint32_t)d; br = (d >> 32) & 1; } zm[2 * H] -= (uint32_t)br; }
  { uint64_t br = 0; for (int i = 0; i < 2 * H; i++) { uint64_t d = (uint64_t)zm[i] - t[2 * H + i] - br; zm[i] = (uint32_t)d; br = (d >> 32) & 1; } zm[2 * H] -= (uint32_t)br; }
  { uint64_t c = 0; for (int i = 0; i <= 2 * H; i++) { c += (uint64_t)t[H + i] + zm[i]; t[H + i] = (uint32_t)c; c >>= 32; }
    for (int i = 3 * H + 1; i < 4 * H; i++) { c += t[i]; t[i] = (uint32_t)c; c >>= 32; } }
#endif
}

// (v + m q) / R for an N-limb integer v (any value below 2^(32N)); result < q + 1 limbs-wise NOT reduced: below 2q
template <class P>
GMSM_HD void fp_redc_half(const uint32_t* v, uint32_t* out) {
  constexpr int N = P::N;
#if defined(GMSM_PTX_PATH) && !defined(GMSM_PORTABLE_MUL)
  uint32_t A[N + 2], B[N + 2];
#pragma unroll
  for (int i = 0; i < N + 2; i++) A[i] = B[i] = 0;
  uint32_t dprev = 0, e0prev = 0;
#pragma unroll
  for (int i = 0; i < N; i++) {
    uint32_t* Ev = (i & 1) ? B : A;
    uint32_t* Od = (i & 1) ? A : B;
    const uint32_t d = (i == 0) ? 0u : Od[1];
    if (i == 0) {
      // row 0 of the CIOS with y_0 = 1: Ev pairs = (v_even, 0), Od pairs = (v_odd, 0)
#pragma unroll
      for (int j = 0; j < N; j += 2) { Ev[j] = v[j]; Ev[j + 1] = 0; Od[j] = v[j + 1]; Od[j + 1] = 0; }
    } else {
      // later rows add nothing: the row's carry-in ripples through Ev, Od is shifted two limbs
      (void)add_cc(e0prev, dprev);
#pragma unroll
      for (int j = 0; j < N; j++) Ev[j] = addc_cc(Ev[j], 0);
      Ev[N] = addc(0, 0);
#pragma unroll
      for (int j = 0; j < N; j++) Od[j] = Od[j + 2];
      Od[N] = 0;
    }
    const uint32_t m = (Ev[0] + d) * invm<P>();
    Ev[0] = mad_lo_cc(modm<P>(0), m, Ev[0]);
    Ev[1] = madc_hi_cc(modm<P>(0), m, Ev[1]);
#pragma unroll
    for (int j = 2; j < N; j += 2) {
      Ev[j] = madc_lo_cc(modm<P>(j), m, Ev[j]);
      Ev[j + 1] = madc_hi_cc(modm<P>(j), m, Ev[j + 1]);
    }
    Ev[N] = addc(Ev[N], 0);
    Od[0] = mad_lo_cc(modm<P>(1), m, Od[0]);
    Od[1] = madc_hi_cc(modm<P>(1), m, Od[1]);
#pragma unroll
    for (int j = 2; j < N; j += 2) {
      Od[j] = madc_lo_cc(modm<P>(j + 1), m, Od[j]);
      Od[j + 1] = madc_hi_cc(modm<P>(j + 1), m, Od[j + 1]);
    }
    GMSM_NO_CARRY();
    e0prev = Ev[0];
    dprev = d;
  }
  (void)add_cc(e0prev, dprev);
  out[0] = addc_cc(A[0], B[1]);
#pragma unroll
  for (int i = 1; i < N - 1; i++) out[i] = addc_cc(A[i], B[i + 1]);
  out[N - 1] = addc(A[N - 1], B[N]);
#else
  uint32_t t[N + 2];
  for (int i = 0; i < N; i++) t[i] = v[i];
  t[N] = t[N + 1] = 0;
  for (int i = 0; i < N; i++) {
    const uint32_t m = t[0] * P::INV;
    uint64_t c = (uint64_t)m * P::mod(0) + t[0];
    c >>= 32;
    for (int j = 1; j < N; j++) {
      c += (uint64_t)m * P::mod(j) + t[j];
      t[j - 1] = (uint32_t)c;
      c >>= 32;
    }
    c += t[N];
    t[N - 1] = (uint32_t)c;
    t[N] = (uint32_t)(c >> 32);
  }
  for (int i = 0; i < N; i++) out[i] = t[i];
#endif
}

// T * R^-1 mod q, fully reduced, for a 2N-limb T < NRED * q * R (redc_half(T_lo) <= q, T_hi < NRED * q: NRED conditional
// subtractions; (NRED + 1) q must fit the limbs)
template <class P, int NRED = 3>
GMSM_HD Fp<P> fp_redc_wide(const uint32_t* t) {
  constexpr int N = P::N;
  uint32_t lo[N];
  fp_redc_half<P>(t, lo);
  Fp<P> r;
#if defined(GMSM_PTX_PATH)
  r.l[0] = add_cc(lo[0], t[N]);
#pragma unroll
  for (int i = 1; i < N - 1; i++) r.l[i] = addc_cc(lo[i], t[N + i]);
  r.l[N - 1] = addc(lo[N - 1], t[2 * N - 1]);
#else
  uint64_t c = 0;
  for (int i = 0; i < N; i++) {
    c += (uint64_t)lo[i] + t[N + i];
    r.l[i] = (uint32_t)c;
    c >>= 32;
  }
#endif
#pragma unroll
  for (int k = 0; k < NRED; k++) fp_reduce_once(r);
  return r;
}

// x * y = REDC(Karatsuba(x, y)): 3 (N/2)^2 + N^2 + N IMAD.WIDE (120 for N = 8 instead of 136); inputs < q, so T < q^2 and one
// conditional subtraction suffices
template <class P>
GMSM_HD Fp<P> fp_mul_karatsuba(const Fp<P>& x, const Fp<P>& y) {
  uint32_t t[2 * P::N];
  mul_wide_karatsuba<P::N>(x.l, y.l, t);
  return fp_redc_wide<P, 1>(t);
}

// x * y through the separated routines (for tests: identical values to fp_mul)
template <class P>
GMSM_HD Fp<P> fp_mul_split(const Fp<P>& x, const Fp<P>& y) {
  uint32_t t[2 * P::N];
  fp_mul_wide<P>(x.l, y.l, t);
  return fp_redc_wide<P>(t);
}

// Montgomery -> canonical: multiply by 1 (fromMont, fr/element.go:593-642)
template <class P>
GMSM_HD Fp<P> fp_from_mont(const Fp<P>& x) {
  Fp<P> o = Fp<P>::zero();
  o.l[0] = 1;
  return fp_mul(x, o);
}

// canonical -> Montgomery (toMont, fp/element.go:782-784)
template <class P>
GMSM_HD Fp<P> fp_to_mont(const Fp<P>& x) {
  Fp<P> r2;
#pragma unroll
  for (int i = 0; i < P::N; i++) r2.l[i] = P::r2(i);
  return fp_mul(x, r2);
}

// x^-1 by Fermat (x^(q-2)); Inverse(0) = 0 like fp/element.go:1170-1172.  Any correct inversion
// is limb-identical to the reference's Pornin GCD since the reduced Montgomery value is unique.
// Kept for the batched-inversion kernels' cross-check; the engine uses fp_inv (binary GCD) below.
template <class P>
GMSM_HD Fp<P> fp_inv_fermat(const Fp<P>& x) {
  constexpr int N = P::N;
  // exponent e = q - 2
  uint32_t e[N];
  {
    uint64_t br = 2;
    for (int i = 0; i < N; i++) {
      uint64_t d = (uint64_t)P::mod(i) - br;
      e[i] = (uint32_t)d;
      br = (d >> 32) & 1;
    }
  }
  Fp<P> acc = Fp<P>::one();
  bool started = false;
  for (int i = 32 * N - 1; i >= 0; i--) {
    if (started) acc = fp_sqr(acc);
    if ((e[i >> 5] >> (i & 31)) & 1) {
      acc = started ? fp_mul(acc, x) : x;
      started = true;
    }
  }
  return acc;
}

// x^-1 by the binary extended Euclidean algorithm on the integer a = x*R mod q (the stored limbs):
//   invariants  x1 * a = u,  x2 * a = v  (mod q);  u, v shrink by halving / subtraction until one of them is 1.
// <= 2 * 32N iterations of shifts and additions on N limbs -- no multiplications -- against the ~1.5 * 32N dependent
// Montgomery products of the Fermat ladder: the inversion at the end of an MSM (FromJacobian, g1.go:150-166) sits on the
// serial tail, where one product costs ~0.5 us of latency.  (The reference uses Pornin's optimised binary GCD,
// fp/element.go:1173-1325; any correct inverse is limb-identical.)  a^-1 = x^-1 R^-1, so two products by R^2 bring the
// result back to Montgomery form.  Inverse(0) = 0.  For a full-width q the bit of x1 + q above the limbs is shifted back in.
template <class P>
GMSM_HD Fp<P> fp_inv(const Fp<P>& x) {
  constexpr int N = P::N;
  if (x.is_zero()) return x;
  uint32_t u[N], v[N], x1[N], x2[N];
  for (int i = 0; i < N; i++) { u[i] = x.l[i]; v[i] = P::mod(i); x1[i] = 0; x2[i] = 0; }
  x1[0] = 1;
  auto is_one = [](const uint32_t* a) { uint32_t o = a[0] ^ 1u; for (int i = 1; i < N; i++) o |= a[i]; return o == 0; };
  // a = (top : a) >> 1 -- top is the bit above the limbs (the carry of y + q for a full-width q, otherwise 0)
  auto shr1 = [](uint32_t* a, uint32_t top) { for (int i = 0; i < N - 1; i++) a[i] = (a[i] >> 1) | (a[i + 1] << 31); a[N - 1] = (a[N - 1] >> 1) | (top << 31); };
  auto add_mod = [](uint32_t* a) { uint64_t c = 0; for (int i = 0; i < N; i++) { c += (uint64_t)a[i] + P::mod(i); a[i] = (uint32_t)c; c >>= 32; } return (uint32_t)c; };
  auto geq = [](const uint32_t* a, const uint32_t* b) { for (int i = N - 1; i >= 0; i--) { if (a[i] != b[i]) return a[i] > b[i]; } return true; };
  auto sub = [](uint32_t* a, const uint32_t* b) { uint64_t br = 0; for (int i = 0; i < N; i++) { uint64_t d = (uint64_t)a[i] - b[i] - br; a[i] = (uint32_t)d; br = (d >> 32) & 1; } return (uint32_t)br; };
  auto halve = [&](uint32_t* w, uint32_t* y) {   // w even: w /= 2, y /= 2 mod q
    shr1(w, 0);
    const uint32_t top = (y[0] & 1u) ? add_mod(y) : 0u;   // y + q < 2q: one bit above the limbs when q fills them (P::FULL)
    shr1(y, top);
  };
  auto sub_mod = [&](uint32_t* a, const uint32_t* b) { if (sub(a, b)) add_mod(a); };   // a = a - b mod q (a, b < q; the wrap is exact)
  while (!is_one(u) && !is_one(v)) {
    while (!(u[0] & 1u)) halve(u, x1);
    while (!(v[0] & 1u)) halve(v, x2);
    if (geq(u, v)) { sub(u, v); sub_mod(x1, x2); } else { sub(v, u); sub_mod(x2, x1); }
  }
  Fp<P> r, r2;
  for (int i = 0; i < N; i++) { r.l[i] = is_one(u) ? x1[i] : x2[i]; r2.l[i] = P::r2(i); }
  return fp_mul(fp_mul(r, r2), r2);
}

// uniform coordinate-field interface (overloaded for Fp2 in fp2.cuh)
template <class P> GMSM_HD Fp<P> f_add(const Fp<P>& a, const Fp<P>& b) { return fp_add(a, b); }
template <class P> GMSM_HD Fp<P> f_sub(const Fp<P>& a, const Fp<P>& b) { return fp_sub(a, b); }
template <class P> GMSM_HD Fp<P> f_mul(const Fp<P>& a, const Fp<P>& b) { return fp_mul(a, b); }
template <class P> GMSM_HD Fp<P> f_sqr(const Fp<P>& a) { return fp_sqr(a); }
template <class P> GMSM_HD Fp<P> f_dot2(const Fp<P>& x, const Fp<P>& y, const Fp<P>& u, const Fp<P>& v) { return fp_dot2(x, y, u, v); }
template <class P> GMSM_HD Fp<P> f_dbl(const Fp<P>& a) { return fp_dbl(a); }
template <class P> GMSM_HD Fp<P> f_neg(const Fp<P>& a) { return fp_neg(a); }
template <class P> GMSM_HD Fp<P> f_inv(const Fp<P>& a) { return fp_inv(a); }

// the prime field a coordinate field is built on (Fp itself here; the Fp2 specialisation is in fp2.cuh)
template <class F> struct base_field;
template <class P> struct base_field<Fp<P>> { using type = Fp<P>; };

}  // namespace gmsm

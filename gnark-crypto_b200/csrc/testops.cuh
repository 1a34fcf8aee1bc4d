// Element-wise test operations (include/gmsm.h GMSM_OP_*), host+device: the same code is run on the GPU
// by k_test_op and on the CPU (portable arithmetic path) by csrc/hostcheck.cpp.
#pragma once
#include "groups.cuh"

namespace gmsm {

// ------------------------------------------------------------------------------------------
template <class T>
GMSM_HD T rd(const uint32_t* p) {
  T r;
  uint32_t* w = reinterpret_cast<uint32_t*>(&r);
  for (int i = 0; i < (int)(sizeof(T) / 4); i++) w[i] = p[i];
  return r;
}
template <class T>
GMSM_HD void wr(uint32_t* p, const T& r) {
  const uint32_t* w = reinterpret_cast<const uint32_t*>(&r);
  for (int i = 0; i < (int)(sizeof(T) / 4); i++) p[i] = w[i];
}

template <class G>
GMSM_HD void test_op_sizes(int op, int* wa, int* wb, int* wo) {
  constexpr int FW = G::F::N;
  constexpr int BW = base_field<typename G::F>::type::N;
  switch (op) {
    case 0: case 1: case 2: *wa = FW; *wb = FW; *wo = FW; break;
    case 3: case 4: case 5: case 6: *wa = FW; *wb = 0; *wo = FW; break;
    case 7: case 8: *wa = 4 * FW; *wb = 2 * FW; *wo = 4 * FW; break;
    case 9: *wa = 4 * FW; *wb = 4 * FW; *wo = 4 * FW; break;
    case 10: *wa = 4 * FW; *wb = 0; *wo = 4 * FW; break;
    case 11: *wa = 4 * FW; *wb = 0; *wo = 2 * FW; break;
    case 12: *wa = G::Fr::N; *wb = 0; *wo = G::Fr::N; break;
    case 13: *wa = 2 * FW; *wb = 2 * FW; *wo = FW; break;
    case 14: *wa = 4 * BW; *wb = 4 * BW; *wo = BW; break;
    default: *wa = *wb = *wo = 0;
  }
}

template <class G>
GMSM_HD void test_op_one(int op, const uint32_t* a, const uint32_t* b, uint32_t* o) {
  using F = typename G::F;
  switch (op) {
    case 0: wr(o, f_mul(rd<F>(a), rd<F>(b))); break;
    case 1: wr(o, f_add(rd<F>(a), rd<F>(b))); break;
    case 2: wr(o, f_sub(rd<F>(a), rd<F>(b))); break;
    case 3: wr(o, f_sqr(rd<F>(a))); break;
    case 4: wr(o, f_neg(rd<F>(a))); break;
    case 5: wr(o, f_dbl(rd<F>(a))); break;
    case 6: wr(o, f_inv(rd<F>(a))); break;
    case 7: case 8: {
      XYZZ<F> p = rd<XYZZ<F>>(a);
      xyzz_add_mixed(p, rd<Affine<F>>(b), op == 8);
      wr(o, p);
    } break;
    case 9: {
      XYZZ<F> p = rd<XYZZ<F>>(a);
      xyzz_add(p, rd<XYZZ<F>>(b));
      wr(o, p);
    } break;
    case 10: wr(o, xyzz_double(rd<XYZZ<F>>(a))); break;
    case 11: wr(o, jac_to_affine(xyzz_to_jac(rd<XYZZ<F>>(a)))); break;
    case 12: wr(o, fp_from_mont(rd<typename G::Fr>(a))); break;
    case 13: wr(o, f_dot2(rd<F>(a), rd<F>(b), rd<F>(a + F::N), rd<F>(b + F::N))); break;   // x y + u v: a = [x | u], b = [y | v]
    case 14: {   // x0 y0 + .. + x3 y3 in the base field: a = x0..x3, b = y0..y3
      using B = typename base_field<F>::type;
      wr(o, fp_dot4(rd<B>(a), rd<B>(b), rd<B>(a + B::N), rd<B>(b + B::N), rd<B>(a + 2 * B::N), rd<B>(b + 2 * B::N), rd<B>(a + 3 * B::N),
                    rd<B>(b + 3 * B::N)));
    } break;
    default: break;
  }
}


}  // namespace gmsm

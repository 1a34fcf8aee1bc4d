// Host orchestration + C ABI (include/gmsm.h) of the B200 MSM engine.
// There is deliberately no CPU fallback: every entry point fails with GMSM_ENODEV / GMSM_ECUDA when
// the device path is unavailable.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <atomic>
#include <condition_variable>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "engine.h"

using namespace gmsm;

// ------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------
static thread_local std::string g_err;
static int g_last_oneshot_launches = 0;

int gmsm::set_err(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}

extern "C" const char* gmsm_last_error(void) { return g_err.c_str(); }
extern "C" int gmsm_last_oneshot_launches(void) { return g_last_oneshot_launches; }
extern "C" const char* gmsm_version(void) { return "gmsm-b200 0.1 (sm_100a)"; }

// ------------------------------------------------------------------------------------------
// per-curve dispatch
// ------------------------------------------------------------------------------------------
static bool curve_info(int curve, CurveInfo* ci) {
  switch (curve) {
    case GMSM_BN254_G1: *ci = {bn254_g1::F::N, bn254_fr::BITS, 4 * bn254_fr::N}; return true;
    case GMSM_BN254_G2: *ci = {bn254_g2::F::N, bn254_fr::BITS, 4 * bn254_fr::N}; return true;
    case GMSM_BLS12381_G1: *ci = {bls12381_g1::F::N, bls12381_fr::BITS, 4 * bls12381_fr::N}; return true;
    case GMSM_BLS12381_G2: *ci = {bls12381_g2::F::N, bls12381_fr::BITS, 4 * bls12381_fr::N}; return true;
    case GMSM_BLS12377_G1: *ci = {bls12377_g1::F::N, bls12377_fr::BITS, 4 * bls12377_fr::N}; return true;
    case GMSM_BLS12377_G2: *ci = {bls12377_g2::F::N, bls12377_fr::BITS, 4 * bls12377_fr::N}; return true;
    case GMSM_SECP256K1_G1: *ci = {secp256k1_g1::F::N, secp256k1_fr::BITS, 4 * secp256k1_fr::N}; return true;
    case GMSM_BW6761_G1: *ci = {bw6761_g1::F::N, bw6761_fr::BITS, 4 * bw6761_fr::N}; return true;
    case GMSM_BW6761_G2: *ci = {bw6761_g2::F::N, bw6761_fr::BITS, 4 * bw6761_fr::N}; return true;
    case GMSM_BLS24315_G1: *ci = {bls24315_g1::F::N, bls24315_fr::BITS, 4 * bls24315_fr::N}; return true;
    case GMSM_BLS24317_G1: *ci = {bls24317_g1::F::N, bls24317_fr::BITS, 4 * bls24317_fr::N}; return true;
    case GMSM_BW6633_G1: *ci = {bw6633_g1::F::N, bw6633_fr::BITS, 4 * bw6633_fr::N}; return true;
    case GMSM_BW6633_G2: *ci = {bw6633_g2::F::N, bw6633_fr::BITS, 4 * bw6633_fr::N}; return true;
  }
  return false;
}

extern "C" size_t gmsm_affine_bytes(gmsm_curve_t c) { CurveInfo ci; return curve_info(c, &ci) ? 8u * ci.coord_words : 0; }
extern "C" size_t gmsm_scalar_bytes(gmsm_curve_t c) { CurveInfo ci; return curve_info(c, &ci) ? (size_t)ci.scalar_bytes : 0; }
extern "C" size_t gmsm_jac_bytes(gmsm_curve_t c) { CurveInfo ci; return curve_info(c, &ci) ? 12u * ci.coord_words : 0; }
extern "C" size_t gmsm_xyzz_bytes(gmsm_curve_t c) { CurveInfo ci; return curve_info(c, &ci) ? 16u * ci.coord_words : 0; }

static const GroupVTable* vtable(int curve) {
  switch (curve) {
    case GMSM_BN254_G1: return &vt_bn254_g1;
    case GMSM_BN254_G2: return &vt_bn254_g2;
    case GMSM_BLS12381_G1: return &vt_bls12381_g1;
    case GMSM_BLS12381_G2: return &vt_bls12381_g2;
    case GMSM_BLS12377_G1: return &vt_bls12377_g1;
    case GMSM_BLS12377_G2: return &vt_bls12377_g2;
    case GMSM_SECP256K1_G1: return &vt_secp256k1_g1;
    case GMSM_BW6761_G1: return &vt_bw6761_g1;
    case GMSM_BW6761_G2: return &vt_bw6761_g2;
    case GMSM_BLS24315_G1: return &vt_bls24315_g1;
    case GMSM_BLS24317_G1: return &vt_bls24317_g1;
    case GMSM_BW6633_G1: return &vt_bw6633_g1;
    case GMSM_BW6633_G2: return &vt_bw6633_g2;
  }
  return nullptr;
}

// ------------------------------------------------------------------------------------------
// window-width model (the reference's bestC, multiexp.go:75-93, minimises (Bits + 1)(n + 2^c)/c over c <= 16 for a CPU whose
// bucket array must stay in cache; the GPU's trade-off is different and is modelled from measurements).
//   T(c) = n * W(c) * e_g(c)  +  tail_g(c)
//   e_g(c)    time per bucket entry (one mixed addition + its share of the digit / sort passes): the measured accumulate rate
//             of the group's kernel (multiplier-pipe bound, DESIGN.md section 5), 1.2 % more per bit of c beyond 17 (the
//             bucket array outgrows L2-friendly sizes), + 9 ps for K1 + the exposed part of the scatter
//   tail_g(c) the n-independent stages -- carry join, bucket reduction (2^(c-1) W buckets: latency-bound below ~10^6 buckets,
//             throughput-bound above), Horner over the windows, normalisation -- read from a table measured per group
//             (profiles/r02_c_sweep_call3.txt: total - accumulate - digits - scatter of a width sweep), because its shape
//             depends on occupancy steps of the tail kernels that no closed form captures
// The table values are milliseconds on a B200 at 1965 MHz; on another part the argmin moves little because both terms scale
// with the same clock.  Validation: profiles/r02_window_model_validation.md (the model's choice is within 2 % of the best
// measured width for every swept configuration).  c can still be forced through gmsm_ctx_create / GMSM_C.
// ------------------------------------------------------------------------------------------
struct WidthModel {
  double add_ns;          // accumulate: ns per mixed addition at c <= 17
  double tail_ms[7];      // tail_g(c) for c = 13 .. 19
  double fixed_ms;        // beyond c = 19: tail = fixed_ms + red19_ms * 2^(c - 19) (the bucket reduction doubles per bit, the carry
  double red19_ms;        //   join / Horner / inversion do not; measured at c = 20, 21); red19_ms = 0: tail_ms[6] * 2^(c - 19)
};
static const WidthModel& width_model(int curve) {
  static const WidthModel bn254_g1 = {0.157, {2.56, 2.43, 2.19, 2.24, 2.41, 3.74, 6.30}, 1.7, 3.0};
  static const WidthModel bls_g1 = {0.366, {5.29, 5.33, 4.42, 4.59, 5.75, 6.88, 8.53}, 2.85, 4.5};
  static const WidthModel bn254_g2 = {0.509, {6.50, 6.37, 5.81, 5.95, 5.70, 9.30, 12.0}, 4.45, 6.67};
  static const WidthModel bls_g2 = {1.300, {13.6, 13.3, 12.2, 12.5, 12.0, 19.6, 25.2}, 0, 0};
  // N4 remainder: fitted from the width sweeps of profiles/r02_n4_new_curves_call11.txt / _call12.txt.  secp256k1: fr.Bits = 256
  // makes the last window narrow for most widths (K1 contention, below).  bw6-761: the 377 doublings of the 24-limb Horner chain alone are ~9 ms.
  static const WidthModel secp256k1_g1 = {0.1755, {2.50, 2.50, 2.95, 3.08, 3.45, 4.17, 5.66}, 2.05, 3.30};
  static const WidthModel bw6761 = {1.63, {16.8, 16.5, 17.7, 19.3, 25.9, 30.2, 46.6}, 13.2, 33.4};
  // 10- and 20-limb groups (bls24-315 / bls24-317 G1, bw6-633): fitted from profiles/r02_n4_more_curves_call13.txt; bw6-633's
  // c = 17 entry absorbs an accumulate that is 6 % slower per addition at that width than at 16 or 18
  static const WidthModel bls24_g1 = {0.255, {3.38, 3.30, 3.31, 3.50, 3.61, 4.95, 6.18}, 2.5, 3.62};
  static const WidthModel bw6633 = {1.08, {13.05, 13.3, 12.4, 13.4, 19.6, 18.9, 28.2}, 9.5, 18.7};
  switch (curve) {
    case GMSM_SECP256K1_G1: return secp256k1_g1;
    case GMSM_BW6761_G1: case GMSM_BW6761_G2: return bw6761;
    case GMSM_BLS24315_G1: case GMSM_BLS24317_G1: return bls24_g1;
    case GMSM_BW6633_G1: case GMSM_BW6633_G2: return bw6633;
    case GMSM_BN254_G1: return bn254_g1;
    case GMSM_BLS12381_G1: case GMSM_BLS12377_G1: return bls_g1;
    case GMSM_BN254_G2: return bn254_g2;
    default: return bls_g2;
  }
}
static double model_ms(int curve, int fr_bits, size_t n, int c) {
  const WidthModel& m = width_model(curve);
  const WindowPlan p = make_plan(fr_bits, c);
  double tail;
  if (c < 13) tail = m.tail_ms[0] * (1.0 + 0.03 * (13 - c));        // more windows: longer Horner / more launches, fewer buckets
  else if (c > 19) tail = m.red19_ms > 0 ? m.fixed_ms + m.red19_ms * (double)(1u << (c - 19))
                                         : m.tail_ms[6] * (double)(1u << (c - 19));  // bucket reduction doubles per bit
  else tail = m.tail_ms[c - 13];
  // a narrow last window puts all its n entries on a handful of buckets: the histogram / rank atomics of K1 serialise on those
  // addresses.  Measured at 2^24 (profiles/r02_n4_new_curves_call11.txt, r02_c20_checks_call15.txt): +5.6 ms with 2 buckets
  // (secp256k1 c = 15, 17), +2.7 ms with 16 (c = 18), +3.8 ms with 64 (bls24-315 c = 19), +3.9 ms with 256 (bls12-381 c = 19),
  // +2.0 ms with 512 (secp256k1 c = 19), nothing from 2^13 buckets on: 0.35 ns per entry up to 4 buckets, 0.2 ns up to 1024.
  // (This is what made c = 19 a poor choice for the 255- / 253-bit curves at 2^24: 13 windows of 20 bits end on a full-width
  // last window and win -- bls12-381 G1 105.0 -> 96.8 ms, bls12-377 G1 117.2 -> 114.2 ms, bn254 G1 at 2^25 86.8 -> 83.4 ms.)
  if (p.nwin > 1 && p.nb_last <= 1024) tail += 1e-6 * (double)n * (p.nb_last <= 4 ? 0.35 : 0.2);
  const double e_ns = m.add_ns * (1.0 + 0.012 * std::max(0, c - 17)) + 0.009;
  return (double)n * p.nwin * e_ns * 1e-6 + tail;
}
// Entries (one per non-zero digit) are numbered with 32-bit indices: a context holds at most max_n * W < MAX_ENTRIES of them.
// With K <= 256 this also keeps the end of the last accumulate chunk, start + K, below 2^32.
static constexpr double MAX_ENTRIES = 4294967000.0;
static bool entries_fit(int fr_bits, size_t capacity, int c) { return (double)capacity * make_plan(fr_bits, c).nwin < MAX_ENTRIES; }

// n: the size the model prices; capacity: the largest n ONE context built with the width has to hold (a pipelined call's largest
// batch, not its total).  Only widths whose capacity * W fits the entry index are candidates: [4, 22] first, then c = 23, 24
// (from n ~ 3.6e8 on the 253..256-bit fields no width up to 22 fits, c = 24 with W = 11 does).  When no width fits, the model's
// unconstrained choice is returned and ctx_create_ex refuses it with the 32-bit-index error.
static int choose_c_for(int curve, int fr_bits, size_t n, size_t capacity) {
  if (const char* e = getenv("GMSM_C")) {
    int c = atoi(e);
    if (c >= 2 && c <= 24) return c;
  }
  auto best_of = [&](int lo, int hi, bool must_fit) {
    double best = 1e300;
    int bc = 0;
    for (int c = lo; c <= hi; c++) {
      if (must_fit && !entries_fit(fr_bits, capacity, c)) continue;
      const double t = model_ms(curve, fr_bits, n, c);
      if (t < best) { best = t; bc = c; }
    }
    return bc;
  };
  if (int c = best_of(4, 22, true)) return c;
  if (int c = best_of(23, 24, true)) return c;
  return best_of(4, 22, false);
}

// window width of the window-table mode: one shared bucket set, so the bucket reduction costs 2^(c-1) * ~3.8
// full-add equivalents ONCE instead of per window, and c can grow until that term meets the W(c)*n accumulate
// term: c = 22 (W = 12) at n = 2^24 for the 253..255-bit scalar fields.  GMSM_TABLE_C forces it.
static int choose_c_tables(int fr_bits, size_t n) {
  if (const char* e = getenv("GMSM_TABLE_C")) {
    int c = atoi(e);
    if (c >= 2 && c <= 24) return c;
  }
  double best = 1e300;
  int bc = 8;
  for (int c = 6; c <= 24; c++) {
    WindowPlan p = make_plan(fr_bits, c);
    double cost = (double)p.nwin * (double)n + (double)std::max(p.nb, p.nb_last) * 3.8 * 1.4;
    if (cost < best) { best = cost; bc = c; }
  }
  return bc;
}

// ------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------
static int ctx_alloc(gmsm_ctx* c) {
  const WindowPlan& p = c->plan;
  const size_t xyzz = 16u * c->ci.coord_words;
  size_t acc = 0;
  const size_t nbp = (size_t)p.nb_total + 1;
  CK(dmalloc(&c->hist, (nbp + 8) * 4, &acc));
  CK(dmalloc(&c->offsets, (nbp + 8) * 4, &acc));
  CK(dmalloc(&c->block_sums, ((nbp + SCAN_TILE - 1) / SCAN_TILE + 8) * 4, &acc));
  const size_t ent = c->max_n * (size_t)p.nwin;
  CK(dmalloc(&c->entries, (ent + 16) * 4, &acc));
  CK(dmalloc(&c->digits, (ent + 16) * 4, &acc));
  CK(dmalloc(&c->ranks, (ent + 16) * 4, &acc));
  CK(dmalloc(&c->buckets, (size_t)p.nb_total * xyzz, &acc));
  // chunks(n) = ceil(n*W / K(n)) <= max(148*512*8 (+slack), ceil(max_n*W/128))  -- see pick_K
  size_t mc = std::max<size_t>(700000, (ent + 127) / 128 + 1);
  c->max_chunks = mc;
  CK(dmalloc(&c->carries[0], mc * xyzz, &acc));
  CK(dmalloc(&c->carry_ids[0], (mc + 8) * 4, &acc));
  if (const char* e = getenv("GMSM_K2_FIRST")) { int v = atoi(e); if (v >= 2 && v <= 64) c->K2_first = (uint32_t)v; }
  const uint32_t k2min = std::min(c->K2, c->K2_first);
  size_t mc2 = (mc + k2min - 1) / k2min;
  CK(dmalloc(&c->carries[1], mc2 * xyzz, &acc));
  CK(dmalloc(&c->carry_ids[1], (mc2 + 8) * 4, &acc));
  uint32_t nbmax = std::max(p.nb, p.nb_last);
  c->seg_L = 32;  // buckets per reduction segment (GMSM_SEG_L to experiment)
  if (c->shared) c->seg_L = 64;   // one window of 2^21 buckets: measured 2.19 ms against 2.69 ms (L = 32) and 3.24 ms (L = 16)
  if (const char* e = getenv(c->shared ? "GMSM_TABLE_SEG_L" : "GMSM_SEG_L")) { int v = atoi(e); if (v >= 2 && v <= 1024) c->seg_L = (uint32_t)v; }
  c->seg_S = (nbmax + c->seg_L - 1) / c->seg_L;
  CK(dmalloc(&c->seg[0], (size_t)c->red_windows() * c->seg_S * xyzz, &acc));
  CK(dmalloc(&c->seg[1], (size_t)c->red_windows() * ((c->seg_S + 15) / 16) * xyzz, &acc));
  if (c->affine) {
    const size_t aff = 8u * c->ci.coord_words, fe = 4u * c->ci.coord_words;
    const size_t m1 = (ent + std::min(nbp, ent)) / 2 + 2, m2 = (m1 + std::min(nbp, m1)) / 2 + 2;
    c->aff_cap1 = m1; c->aff_cap2 = m2;
    c->aff_tcap = std::max<size_t>(700000, m1 / 128 + 64);
    CK(dmalloc(&c->aff_buf[0], m1 * aff, &acc));
    CK(dmalloc(&c->aff_buf[1], m2 * aff, &acc));
    CK(dmalloc(&c->aff_pref, m1 * fe, &acc));
    CK(dmalloc(&c->aff_totals, c->aff_tcap * fe, &acc));
    CK(dmalloc(&c->aff_ps, c->aff_tcap * fe, &acc));
    CK(dmalloc(&c->aff_bp, 3 * (c->aff_tcap / 1024 + 8) * fe, &acc));
    CK(dmalloc(&c->aff_off[0], (nbp + 8) * 4, &acc));
    CK(dmalloc(&c->aff_off[1], (nbp + 8) * 4, &acc));
    CK(dmalloc(&c->aff_counts, (nbp + 8) * 4, &acc));
    CK(dmalloc(&c->aff_maxlen, 16, &acc));
    CK(cudaMallocHost((void**)&c->aff_maxlen_host, 16));
  }
  CK(dmalloc(&c->win_partials, (size_t)p.nwin * xyzz, &acc));
  CK(dmalloc(&c->fin_scratch, (size_t)p.nwin * xyzz, &acc));
  c->ws_bytes = acc;
  for (int i = 0; i < 9; i++) CK(cudaEventCreate(&c->ev[i]));
  CK(cudaStreamCreateWithFlags(&c->aux, cudaStreamNonBlocking));
  for (int i = 0; i < 2; i++) CK(cudaEventCreateWithFlags(&c->ev_split[i], cudaEventDisableTiming));
  CK(cudaEventCreateWithFlags(&c->ev_done, cudaEventDisableTiming));
  return GMSM_OK;
}

// Point gathers are 64-byte random reads: while an engine context lives on a device, L2 is kept from promoting them to
// 128-byte fetches (measured: DRAM traffic of the bucket pass 32.4 -> 17.2 GB).  The limit is a per-device setting of the
// whole process, so it is reference-counted and the previous value restored when the last context of the device goes away
// (GMSM_L2_FETCH=0 leaves the limit alone).
static std::mutex g_l2_mu;
static std::map<int, std::pair<int, size_t>> g_l2_state;   // device -> (live contexts, previous limit)
static void l2_granularity_acquire(int device) {
  if (const char* e = getenv("GMSM_L2_FETCH")) if (atoi(e) == 0) return;
  std::lock_guard<std::mutex> lk(g_l2_mu);
  auto& st = g_l2_state[device];
  if (st.first++ == 0) {
    size_t prev = 0;
    if (cudaDeviceGetLimit(&prev, cudaLimitMaxL2FetchGranularity) != cudaSuccess) { cudaGetLastError(); prev = 0; }
    st.second = prev;
    if (cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, 32) != cudaSuccess) cudaGetLastError();
  }
}
static void l2_granularity_release(int device) {
  if (const char* e = getenv("GMSM_L2_FETCH")) if (atoi(e) == 0) return;
  std::lock_guard<std::mutex> lk(g_l2_mu);
  auto it = g_l2_state.find(device);
  if (it == g_l2_state.end() || it->second.first == 0) return;
  if (--it->second.first == 0 && it->second.second)
    if (cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, it->second.second) != cudaSuccess) cudaGetLastError();
}

static void ctx_free(gmsm_ctx* c) {
  cudaSetDevice(c->device);
  cudaFree(c->hist); cudaFree(c->offsets); cudaFree(c->block_sums); cudaFree(c->entries); cudaFree(c->digits); cudaFree(c->ranks); cudaFree(c->buckets2); cudaFree(c->buckets);
  for (int i = 0; i < 2; i++) { cudaFree(c->carries[i]); cudaFree(c->carry_ids[i]); cudaFree(c->seg[i]); }
  cudaFree(c->win_partials); cudaFree(c->fin_scratch);
  for (int i = 0; i < 2; i++) { cudaFree(c->aff_buf[i]); cudaFree(c->aff_off[i]); }
  cudaFree(c->aff_pref); cudaFree(c->aff_totals); cudaFree(c->aff_ps); cudaFree(c->aff_bp); cudaFree(c->aff_counts);
  cudaFree(c->aff_maxlen);
  if (c->aff_maxlen_host) cudaFreeHost(c->aff_maxlen_host);
  for (int i = 0; i < 9; i++) if (c->ev[i]) cudaEventDestroy(c->ev[i]);
  for (int i = 0; i < 2; i++) if (c->ev_split[i]) cudaEventDestroy(c->ev_split[i]);
  if (c->aux) cudaStreamDestroy(c->aux);
  if (c->ev_done) cudaEventDestroy(c->ev_done);
  l2_granularity_release(c->device);
}

static gmsm_ctx* ctx_create_ex(gmsm_curve_t curve, size_t max_n, int c, int device, bool shared);
extern "C" gmsm_ctx_t* gmsm_ctx_create(gmsm_curve_t curve, size_t max_n, int c, int device) {
  return ctx_create_ex(curve, max_n, c, device, false);
}
extern "C" gmsm_ctx_t* gmsm_ctx_create_tables(gmsm_curve_t curve, size_t max_n, int c, int device) {
  return ctx_create_ex(curve, max_n, c, device, true);
}

static gmsm_ctx* ctx_create_ex(gmsm_curve_t curve, size_t max_n, int c, int device, bool shared) {
  CurveInfo ci;
  if (!curve_info(curve, &ci)) { set_err(GMSM_EINVAL, "unknown curve id %d", (int)curve); return nullptr; }
  if (c != 0 && (c < 2 || c > 24)) { set_err(GMSM_EINVAL, "window width c=%d out of range [2,24]", c); return nullptr; }
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) { set_err(GMSM_ENODEV, "no CUDA device (%s); this engine has no CPU fallback", cudaGetErrorString(e)); return nullptr; }
  if (device < 0 || device >= ndev) { set_err(GMSM_EINVAL, "device %d out of range (%d devices)", device, ndev); return nullptr; }
  if (cudaSetDevice(device) != cudaSuccess) { set_err(GMSM_ECUDA, "cudaSetDevice(%d) failed", device); return nullptr; }
  if (max_n == 0) max_n = 1;
  l2_granularity_acquire(device);
  gmsm_ctx* ctx = new gmsm_ctx();
  ctx->curve = curve;
  ctx->device = device;
  ctx->max_n = max_n;
  ctx->ci = ci;
  if (c == 0) c = shared ? choose_c_tables(ci.fr_bits, max_n) : choose_c_for(curve, ci.fr_bits, max_n, max_n);
  ctx->shared = shared;
  // bucket accumulation: extended-Jacobian segmented reduction by default (INT-multiplier bound at 89 % of the
  // pipe); GMSM_AFFINE=1 selects the batch-affine tree (fewer multiplies, but 3x the HBM traffic: measured
  // 46.3 ms vs 42.1 ms at bn254 G1 n=2^24, profiles/r01_ncu_affine_*).
  ctx->affine = false;
  if (const char* e = getenv("GMSM_AFFINE")) ctx->affine = atoi(e) != 0;
  if (shared) ctx->affine = false;   // the window-table mode has one accumulation path
  if (const char* e = getenv("GMSM_TABLE_PASSES")) { int v = atoi(e); if (v >= 1 && v <= 256) ctx->table_passes = v; }
  // lane-parallel tail kernels (csrc/quad.cuh), default off: measured slower for the 8- and 12-limb groups (DESIGN.md section 3).
  // bw6-761 (24 limbs: one field product is ~9x bn254's, the serial Horner chain ~10 ms) takes them for the Horner / inversion
  // kernel and for small bucket reductions: 2^18 28.6 -> 27.3 ms, 2^14 17.3 -> 14.8 ms; large reductions stay one thread per
  // segment (2^22: 176.6 vs 186.0 ms with quads everywhere) -- profiles/r02_n4_new_curves_call12.txt
  // (bw6-633, 20 limbs: 2^22 102.6 -> 101.5 ms, 2^18 18.2 -> 17.4 ms, profiles/r02_n4_model_checks_call14.txt)
  if (curve == GMSM_BW6761_G1 || curve == GMSM_BW6761_G2 || curve == GMSM_BW6633_G1 || curve == GMSM_BW6633_G2) {
    ctx->quad_mode = 1;
    ctx->quad_max_items = 20000;
  }
  if (const char* e = getenv("GMSM_QUAD")) { ctx->quad_mode = atoi(e); ctx->quad_max_items = (size_t)1 << 40; }
  if (const char* e = getenv("GMSM_QUAD_MAX")) { long v = atol(e); if (v >= 0) ctx->quad_max_items = (size_t)v; }
  if (const char* e = getenv("GMSM_SPLIT_W")) { int v = atoi(e); if (v >= 1 && v <= 64) ctx->split_w = ctx->split_tab = v; }
  ctx->plan = make_plan(ci.fr_bits, c);
  if (shared) ctx->plan.nb_total = std::max(ctx->plan.nb, ctx->plan.nb_last);   // one bucket set for all windows
  if ((double)max_n * ctx->plan.nwin >= MAX_ENTRIES) {
    set_err(GMSM_EINVAL, "n*W = %zu*%d does not fit the 32-bit entry index; shard the MSM", max_n, ctx->plan.nwin);
    l2_granularity_release(device);
    delete ctx;
    return nullptr;
  }
  if (max_n > (1ull << 31) - 1) { set_err(GMSM_EINVAL, "n too large"); l2_granularity_release(device); delete ctx; return nullptr; }
  if (ctx_alloc(ctx) != GMSM_OK) { ctx_free(ctx); delete ctx; return nullptr; }
  return ctx;
}

extern "C" void gmsm_ctx_destroy(gmsm_ctx_t* ctx) {
  if (!ctx) return;
  ctx_free(ctx);
  delete ctx;
}
extern "C" int gmsm_ctx_window_bits(const gmsm_ctx_t* ctx) { return ctx ? ctx->plan.c : 0; }
extern "C" int gmsm_ctx_num_windows(const gmsm_ctx_t* ctx) { return ctx ? ctx->plan.nwin : 0; }
extern "C" size_t gmsm_ctx_workspace_bytes(const gmsm_ctx_t* ctx) { return ctx ? ctx->ws_bytes : 0; }
extern "C" int gmsm_ctx_last_launches(const gmsm_ctx_t* ctx) { return ctx ? ctx->last_launches : 0; }
extern "C" void gmsm_ctx_set_profiling(gmsm_ctx_t* ctx, int on) { if (ctx) ctx->profiling = on != 0; }
extern "C" int gmsm_ctx_last_stage_ms(gmsm_ctx_t* ctx, float out_ms[8]) {
  if (!ctx || !ctx->have_stage) return set_err(GMSM_EINVAL, "no profiled call recorded");
  cudaSetDevice(ctx->device);
  CK(cudaEventSynchronize(ctx->ev[8]));
  float tot = 0;
  for (int i = 0; i < 7; i++) {
    CK(cudaEventElapsedTime(&out_ms[i], ctx->ev[i], ctx->ev[i + 1]));
  }
  CK(cudaEventElapsedTime(&tot, ctx->ev[0], ctx->ev[7]));
  out_ms[7] = tot;
  return GMSM_OK;
}

// Device-level entry points share one workspace per context and are asynchronous: `CtxCall` holds the context mutex while
// a call is ENQUEUED and chains the calls on the GPU through ctx->ev_done (the call's stream first waits for the previous
// call's completion event, and records it again at the end), so that calls issued from different streams or threads run
// one after the other instead of overlapping on hist / digits / entries / buckets / carries (ADVICE r01).
struct CtxCall {
  gmsm_ctx* c;
  cudaStream_t st;
  std::unique_lock<std::mutex> lk;
  CtxCall(gmsm_ctx* ctx, cudaStream_t s) : c(ctx), st(s), lk(ctx->mu) {}
  int begin() {
    CK(cudaSetDevice(c->device));
    CK(cudaStreamWaitEvent(st, c->ev_done, 0));
    return GMSM_OK;
  }
  ~CtxCall() { cudaEventRecord(c->ev_done, st); }
};

extern "C" int gmsm_ctx_window_sums_device(gmsm_ctx_t* ctx, const void* d_points, const void* d_scalars, size_t n,
                                           void* d_partials, void* stream) {
  if (!ctx) return set_err(GMSM_EINVAL, "null ctx");
  if (ctx->shared) return set_err(GMSM_EINVAL, "window-table context: use gmsm_ctx_msm_tables_device");
  if (n > ctx->max_n) return set_err(GMSM_EINVAL, "n=%zu exceeds ctx capacity %zu", n, ctx->max_n);
  CtxCall call(ctx, (cudaStream_t)stream);
  if (int rc0 = call.begin()) return rc0;
  int rc = GMSM_OK;
  rc = vtable(ctx->curve)->window_sums(ctx, d_points, d_scalars, n, d_partials, (cudaStream_t)stream);
  if (rc == GMSM_OK && ctx->profiling) {
    cudaEventRecord(ctx->ev[7], (cudaStream_t)stream);
    cudaEventRecord(ctx->ev[8], (cudaStream_t)stream);
    ctx->have_stage = true;
  }
  return rc;
}

extern "C" int gmsm_ctx_finalize_device(gmsm_ctx_t* ctx, const void* d_partials, int nranks, void* d_out_jac,
                                        void* stream) {
  if (!ctx) return set_err(GMSM_EINVAL, "null ctx");
  if (nranks < 1) return set_err(GMSM_EINVAL, "nranks must be >= 1");
  CtxCall call(ctx, (cudaStream_t)stream);
  if (int rc0 = call.begin()) return rc0;
  int rc = GMSM_OK;
  rc = vtable(ctx->curve)->finalize(ctx, d_partials, nranks, d_out_jac, (cudaStream_t)stream);
  return rc;
}

extern "C" int gmsm_ctx_msm_device(gmsm_ctx_t* ctx, const void* d_points, const void* d_scalars, size_t n,
                                   void* d_out_jac, void* stream) {
  if (!ctx) return set_err(GMSM_EINVAL, "null ctx");
  if (ctx->shared) return set_err(GMSM_EINVAL, "window-table context: use gmsm_ctx_msm_tables_device");
  if (n > ctx->max_n) return set_err(GMSM_EINVAL, "n=%zu exceeds ctx capacity %zu", n, ctx->max_n);
  CtxCall call(ctx, (cudaStream_t)stream);
  if (int rc0 = call.begin()) return rc0;
  int rc = GMSM_OK;
  cudaStream_t st = (cudaStream_t)stream;
  rc = vtable(ctx->curve)->window_sums(ctx, d_points, d_scalars, n, ctx->win_partials, st);
  if (rc != GMSM_OK) return rc;
  rc = vtable(ctx->curve)->finalize(ctx, ctx->win_partials, 1, d_out_jac, st);
  if (rc != GMSM_OK) return rc;
  ctx->last_launches += 1;
  if (ctx->profiling) {
    cudaEventRecord(ctx->ev[7], st);
    cudaEventRecord(ctx->ev[8], st);
    ctx->have_stage = true;
  }
  return GMSM_OK;
}

// make the device that owns a device pointer current (entry points that take raw device pointers and no context:
// a process driving several GPUs must not depend on the caller's current device)
static int set_device_of(const void* dptr) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, dptr) == cudaSuccess && (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged)) {
    CK(cudaSetDevice(a.device));
  } else {
    cudaGetLastError();
  }
  return GMSM_OK;
}

// ---- window tables (device level) ----
extern "C" int gmsm_tables_build_device(gmsm_curve_t curve, int c, const void* d_points, size_t n, void* d_table,
                                        size_t row_stride, void* stream) {
  CurveInfo ci;
  if (!curve_info(curve, &ci)) return set_err(GMSM_EINVAL, "unknown curve id %d", (int)curve);
  if (c < 2 || c > 24) return set_err(GMSM_EINVAL, "window width c=%d out of range [2,24]", c);
  if (row_stride < n) return set_err(GMSM_EINVAL, "row_stride %zu < n %zu", row_stride, n);
  const WindowPlan p = make_plan(ci.fr_bits, c);
  if ((double)row_stride * p.nwin >= 2147483000.0)
    return set_err(GMSM_EINVAL, "row_stride*W = %zu*%d does not fit the 31-bit table index; shard the bases", row_stride, p.nwin);
  if (n == 0) return GMSM_OK;
  if (int rc = set_device_of(d_table)) return rc;
  const size_t ab = 8u * ci.coord_words;
  cudaStream_t st = (cudaStream_t)stream;
  if (d_table != d_points) CK(cudaMemcpyAsync(d_table, d_points, n * ab, cudaMemcpyDeviceToDevice, st));
  for (int j = 1; j < p.nwin; j++) {
    if (int rc = vtable(curve)->table_level((const char*)d_table + (size_t)(j - 1) * row_stride * ab, n, c,
                                            (char*)d_table + (size_t)j * row_stride * ab, st)) return rc;
  }
  return GMSM_OK;
}

extern "C" int gmsm_ctx_msm_tables_device(gmsm_ctx_t* ctx, const void* d_table, size_t row_stride, size_t offset,
                                          const void* d_scalars, size_t n, void* d_out_jac, void* stream) {
  if (!ctx) return set_err(GMSM_EINVAL, "null ctx");
  if (!ctx->shared) return set_err(GMSM_EINVAL, "context was not created with gmsm_ctx_create_tables");
  if (n > ctx->max_n) return set_err(GMSM_EINVAL, "n=%zu exceeds ctx capacity %zu", n, ctx->max_n);
  if (offset > row_stride || n > row_stride - offset) return set_err(GMSM_EINVAL, "len(points) != len(scalars)");
  if ((double)row_stride * ctx->plan.nwin >= 2147483000.0) return set_err(GMSM_EINVAL, "row_stride*W does not fit the 31-bit table index");
  CtxCall call(ctx, (cudaStream_t)stream);
  if (int rc0 = call.begin()) return rc0;
  cudaStream_t st = (cudaStream_t)stream;
  ctx->tab_stride = (uint32_t)row_stride;
  const size_t ab = 8u * ctx->ci.coord_words;
  int rc = vtable(ctx->curve)->window_sums(ctx, (const char*)d_table + offset * ab, d_scalars, n, ctx->win_partials, st);
  if (rc != GMSM_OK) return rc;
  rc = vtable(ctx->curve)->finalize(ctx, ctx->win_partials, 1, d_out_jac, st);
  if (rc != GMSM_OK) return rc;
  ctx->last_launches += 1;
  if (ctx->profiling) {
    cudaEventRecord(ctx->ev[7], st);
    cudaEventRecord(ctx->ev[8], st);
    ctx->have_stage = true;
  }
  return GMSM_OK;
}

// ------------------------------------------------------------------------------------------
// host staging: pageable caller memory -> pinned ring -> device
// ------------------------------------------------------------------------------------------
// A Go caller hands over ordinary (pageable) slices (SURVEY.md section 8b: cgo pins them only for the duration of the call and
// the library must not keep them).  cudaMemcpyAsync from pageable memory is staged by the driver through one bounce buffer,
// synchronously on the calling thread, at a fraction of the PCIe rate.  The library therefore stages such buffers itself:
// a few host threads copy 32 MiB pieces (in 2 MiB parts) into a ring of pinned slots, each slot is sent with a true asynchronous H2D copy as
// soon as it is full, and the calling thread moves on to fill the next slot -- memcpy, PCIe and the GPU's bucket pass of
// the previous batch all overlap.  Buffers that are already pinned / registered (cudaPointerGetAttributes) skip the ring.
class CopyPool {
 public:
  static CopyPool& get() {
    static CopyPool* p = new CopyPool();   // leaked on purpose: worker threads must not be joined from a static destructor
    return *p;
  }
  // dst[0..n) = src[0..n), cut into 1 MiB parts on a queue shared by all callers; the caller works on the queue too and
  // returns when ITS parts are done.  Concurrent calls (several MultiExp at once) interleave their parts.
  void copy(char* dst, const char* src, size_t n) {
    if (nthreads_ <= 1 || n < (size_t)(2 << 20)) { memcpy(dst, src, n); return; }
    Job job;
    job.remaining.store((int)((n + PART - 1) / PART));
    {
      std::lock_guard<std::mutex> lk(mu_);
      for (size_t off = 0; off < n; off += PART) q_.push_back(Part{dst + off, src + off, std::min(PART, n - off), &job});
    }
    cv_work_.notify_all();
    for (;;) {
      Part p;
      {
        std::lock_guard<std::mutex> lk(mu_);
        if (q_.empty()) break;
        p = q_.front();
        q_.pop_front();
      }
      run(p);
    }
    std::unique_lock<std::mutex> lk(job.mu);
    job.cv.wait(lk, [&] { return job.remaining.load() == 0; });
  }
  int threads() const { return nthreads_; }

 private:
  static constexpr size_t PART = 2 << 20;
  struct Job {
    std::atomic<int> remaining{0};
    std::mutex mu;
    std::condition_variable cv;
  };
  struct Part {
    char* d;
    const char* s;
    size_t n;
    Job* job;
  };
  CopyPool() {
    int hw = (int)std::thread::hardware_concurrency();
    nthreads_ = std::max(1, std::min(16, hw / 4));
    if (const char* e = getenv("GMSM_COPY_THREADS")) { int v = atoi(e); if (v >= 1 && v <= 64) nthreads_ = v; }
    for (int i = 1; i < nthreads_; i++) std::thread([this] { loop(); }).detach();
  }
  static void run(const Part& p) {
    memcpy(p.d, p.s, p.n);
    if (p.job->remaining.fetch_sub(1) == 1) {
      std::lock_guard<std::mutex> lk(p.job->mu);   // (the waiter holds job.mu while it checks: no lost wake-up, no use after free)
      p.job->cv.notify_all();
    }
  }
  void loop() {
    for (;;) {
      Part p;
      {
        std::unique_lock<std::mutex> lk(mu_);
        cv_work_.wait(lk, [&] { return !q_.empty(); });
        p = q_.front();
        q_.pop_front();
      }
      run(p);
    }
  }
  int nthreads_ = 1;
  std::mutex mu_;
  std::condition_variable cv_work_;
  std::deque<Part> q_;
};

struct Stager {
  static constexpr size_t SLOT = 32u << 20;
  static constexpr int NSLOT = 4;
  char* slot[NSLOT] = {};
  cudaEvent_t ev[NSLOT] = {};
  bool used[NSLOT] = {};
  int next = 0;
  int init() {
    if (slot[0]) return GMSM_OK;
    for (int i = 0; i < NSLOT; i++) {
      CK(cudaMallocHost((void**)&slot[i], SLOT));
      CK(cudaEventCreateWithFlags(&ev[i], cudaEventDisableTiming));
    }
    return GMSM_OK;
  }
  void release() {
    for (int i = 0; i < NSLOT; i++) {
      if (slot[i]) cudaFreeHost(slot[i]);
      if (ev[i]) cudaEventDestroy(ev[i]);
      slot[i] = nullptr; ev[i] = nullptr; used[i] = false;
    }
  }
  // pageable src -> device dst on stream st through the ring
  int copy(void* dst, const void* src, size_t bytes, cudaStream_t st) {
    if (int rc = init()) return rc;
    const char* s = reinterpret_cast<const char*>(src);
    char* d = reinterpret_cast<char*>(dst);
    for (size_t off = 0; off < bytes; off += SLOT) {
      const size_t len = std::min(SLOT, bytes - off);
      const int k = next;
      next = (next + 1) % NSLOT;
      if (used[k]) CK(cudaEventSynchronize(ev[k]));   // the slot's previous H2D has left the host buffer
      CopyPool::get().copy(slot[k], s + off, len);
      CK(cudaMemcpyAsync(d + off, slot[k], len, cudaMemcpyHostToDevice, st));
      CK(cudaEventRecord(ev[k], st));
      used[k] = true;
    }
    return GMSM_OK;
  }
};

// is this host pointer pinned (cudaMallocHost / cudaHostRegister) or managed, i.e. safe for a truly asynchronous copy?
static bool host_pointer_is_pinned(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeManaged;
}

// ------------------------------------------------------------------------------------------
// resident bases + one-shot host API
// ------------------------------------------------------------------------------------------
// A pipelined MSM over host scalars (and optionally host points): the inputs are cut into S contiguous
// batches; batch k+1 crosses PCIe on the copy stream while batch k runs K1..K2b on the compute stream,
// every batch accumulating into the same bucket array (rmw); one bucket reduction + finalize at the end.
struct Pipeline {
  int curve = 0, device = 0;
  gmsm_ctx* ctx = nullptr;
  void* d_scalars = nullptr;
  size_t scal_cap = 0;
  void* d_partials = nullptr;
  int partials_cap = 0;
  void* d_out = nullptr;
  cudaStream_t copy_st = nullptr, comp_st = nullptr;
  cudaEvent_t ev[16] = {};
  int last_launches = 0;
  // window-table mode (gmsm_bases_precompute): d_points of pipeline_run is then the table, row stride tab_stride
  bool tables = false;
  size_t tab_stride = 0;
  int tab_c = 0;
  Stager stager;          // pinned ring for pageable caller buffers
  int last_staged = 0;    // 1 if the last call went through the ring
};

static int pipeline_init(Pipeline& P, int curve, int device) {
  if (P.copy_st) return GMSM_OK;
  P.curve = curve; P.device = device;
  CK(cudaStreamCreateWithFlags(&P.copy_st, cudaStreamNonBlocking));
  CK(cudaStreamCreateWithFlags(&P.comp_st, cudaStreamNonBlocking));
  for (int i = 0; i < 16; i++) CK(cudaEventCreateWithFlags(&P.ev[i], cudaEventDisableTiming));
  CK(cudaMalloc(&P.d_out, 512));
  return GMSM_OK;
}

static void pipeline_free(Pipeline& P) {
  if (P.ctx) gmsm_ctx_destroy(P.ctx);
  P.stager.release();
  cudaFree(P.d_scalars); cudaFree(P.d_partials); cudaFree(P.d_out);
  if (P.copy_st) cudaStreamDestroy(P.copy_st);
  if (P.comp_st) cudaStreamDestroy(P.comp_st);
  for (int i = 0; i < 16; i++) if (P.ev[i]) cudaEventDestroy(P.ev[i]);
  P = Pipeline();
}

// batches of a pipelined call over n inputs: batch k is [bstart[k], bstart[k+1]), returns their number.  resident: the points
// are already on the device (only the scalars cross PCIe).
static int plan_batches(size_t n, bool resident, size_t bstart[17]) {
  // batch sizes grow geometrically (1/16, 1/8, 3/16, 1/4, 3/8 of n): the first copy is short, and since the
  // GPU consumes a batch more slowly than PCIe delivers the next, every later copy hides under compute
  static const int FR5[5] = {1, 2, 3, 4, 6};   // sixteenths
  int nch = (n >= (1u << 21)) ? 5 : ((n >= (1u << 18)) ? 2 : 1);
  if (const char* e = getenv("GMSM_CHUNKS")) { int v = atoi(e); if (v >= 1 && v <= 16) nch = v; }
  if ((size_t)nch > n) nch = 1;
  // GMSM_SCHEDULE="1,2,3,5,8": explicit batch weights (experiments; overrides the counts above for n >= 2^18)
  int wts[16], wsum = 0, nw = 0;
  if (resident && n >= (1u << 21) && !getenv("GMSM_CHUNKS")) {
    // resident bases: only the scalars (32 B each) cross PCIe, a third of the one-shot volume, so three batches are
    // enough to hide the copies and every batch less saves its bucket merge + carry join (~1.1 ms each; measured
    // profiles/r01_e2e_schedule_sweep_v15.txt: 4 batches 51.3 ms, 5 batches 52.2 ms at bn254 G1 2^24)
    wts[0] = 1; wts[1] = 3; wts[2] = 9; nw = 3; wsum = 13; nch = 3;
  }
  if (const char* e = getenv("GMSM_SCHEDULE")) {
    nw = 0; wsum = 0;
    if (n >= (1u << 18)) {
      for (const char* q = e; *q && nw < 16;) {
        char* end = nullptr;
        long v = strtol(q, &end, 10);
        if (end == q || v < 1 || v > 1000) break;
        wts[nw++] = (int)v; wsum += (int)v;
        q = (*end == ',') ? end + 1 : end;
      }
      if (nw >= 1) nch = nw;
    }
  }
  bstart[0] = 0;
  for (int k = 1; k <= nch; k++) {
    if (nw >= 1) { long acc = 0; for (int u = 0; u < k; u++) acc += wts[u]; bstart[k] = (k == nch) ? n : (size_t)((double)n * acc / wsum); }
    else if (nch == 5) { int acc16 = 0; for (int u = 0; u < k; u++) acc16 += FR5[u]; bstart[k] = (k == nch) ? n : (n / 16) * acc16; }
    else bstart[k] = (k == nch) ? n : (n / nch) * k;
  }
  return nch;
}
static size_t largest_batch(const size_t bstart[17], int nch) {
  size_t nc = 0;
  for (int k = 0; k < nch; k++) nc = std::max(nc, bstart[k + 1] - bstart[k]);
  return nc;
}
static size_t largest_batch(size_t n, bool resident) {
  size_t bstart[17];
  return largest_batch(bstart, plan_batches(n, resident, bstart));
}

// d_points: device buffer holding (resident) or receiving (h_points != nullptr) the n points
// c_force = 0: window width from n; otherwise the given width (all shards of a multi-device call must share
// one window plan).  h_partials != nullptr: stop after the bucket reduction and return the W window partials
// (host copy) instead of the finalized point.
static int pipeline_run(Pipeline& P, void* d_points, const uint64_t* h_points, const uint64_t* h_scalars, size_t n,
                        uint64_t* out_jac, int c_force = 0, void* h_partials = nullptr) {
  CurveInfo ci;
  curve_info(P.curve, &ci);
  const size_t sb = (size_t)ci.scalar_bytes;
  const size_t ab = 8u * ci.coord_words, xb = 16u * ci.coord_words, jb = 12u * ci.coord_words;
  CK(cudaSetDevice(P.device));
  size_t bstart[17];
  const int nch = plan_batches(n, h_points == nullptr, bstart);
  const size_t nc = largest_batch(bstart, nch);
  if (P.scal_cap < n || P.scal_cap > 4 * n + 1024) {
    cudaFree(P.d_scalars); P.d_scalars = nullptr; P.scal_cap = 0;
    CK(cudaMalloc(&P.d_scalars, n * (size_t)ci.scalar_bytes));
    P.scal_cap = n;
  }
  // window width from the TOTAL size (all batches share one bucket array); workspace sized for one batch
  const int c = P.tables ? P.tab_c : (c_force ? c_force : choose_c_for(P.curve, ci.fr_bits, n, nc));
  if (!P.ctx || P.ctx->max_n < nc || P.ctx->max_n > 4 * nc + 1024 || P.ctx->plan.c != c || P.ctx->shared != P.tables) {
    if (P.ctx) { gmsm_ctx_destroy(P.ctx); P.ctx = nullptr; }
    P.ctx = ctx_create_ex((gmsm_curve_t)P.curve, nc, c, P.device, P.tables);
    if (!P.ctx) return GMSM_ECUDA;
  }
  P.ctx->tab_stride = (uint32_t)P.tab_stride;
  const int npart = P.ctx->red_windows();   // partials per batch / per call: W, or 1 in window-table mode
  if (P.partials_cap < nch * npart) {
    cudaFree(P.d_partials); P.d_partials = nullptr;
    CK(cudaMalloc(&P.d_partials, (size_t)nch * npart * xb));
    P.partials_cap = nch * npart;
  }
  const GroupVTable* vt = vtable(P.curve);
  const char* hp = reinterpret_cast<const char*>(h_points);
  const char* hs = reinterpret_cast<const char*>(h_scalars);
  // the batch-affine path keeps per-batch partials instead (and cannot return per-device partials)
  const bool shared_buckets = !P.ctx->affine;
  if (h_partials && !shared_buckets) return set_err(GMSM_EINVAL, "multi-device calls need the default accumulation mode");
  if (shared_buckets && nch > 1 && !P.ctx->buckets2) {
    CK(cudaMalloc(&P.ctx->buckets2, (size_t)P.ctx->plan.nb_total * xb));
  }
  int launches = 0;
  std::lock_guard<std::mutex> lk(P.ctx->mu);
  // Every exit path -- success or error -- leaves with the copy, compute and auxiliary streams drained: the caller's host
  // buffers (and, on the next call, this pipeline's device buffers) may be reused or freed as soon as we return
  // (SURVEY.md section 8b "finish all reads before returning").
  struct Drain {
    Pipeline& P;
    ~Drain() {
      cudaStreamSynchronize(P.copy_st);
      cudaStreamSynchronize(P.comp_st);
      if (P.ctx && P.ctx->aux) cudaStreamSynchronize(P.ctx->aux);
    }
  } drain{P};
  // pageable caller buffers go through the pinned ring (GMSM_STAGING=0: hand them to cudaMemcpyAsync as they are)
  bool staging = true;
  if (const char* e = getenv("GMSM_STAGING")) staging = atoi(e) != 0;
  const bool stage_scalars = staging && n * (size_t)ci.scalar_bytes >= (1u << 20) && !host_pointer_is_pinned(hs);
  const bool stage_points = staging && hp && n * ab >= (1u << 20) && !host_pointer_is_pinned(hp);
  P.last_staged = (stage_scalars || stage_points) ? 1 : 0;
  auto h2d = [&](void* dst, const char* src, size_t bytes, bool staged) -> int {
    if (staged) return P.stager.copy(dst, src, bytes, P.copy_st);
    CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, P.copy_st));
    return GMSM_OK;
  };
  int fault_after = -1;   // test hook: fail after the given batch has been enqueued (the streams are then busy)
  if (const char* e = getenv("GMSM_FAULT_AFTER_BATCH")) fault_after = atoi(e);
  for (int k = 0; k < nch; k++) {
    const size_t off = bstart[k];
    const size_t m = bstart[k + 1] - off;
    if (int rc = h2d((char*)P.d_scalars + off * sb, hs + off * sb, m * sb, stage_scalars)) return rc;
    if (hp) if (int rc = h2d((char*)d_points + off * ab, hp + off * ab, m * ab, stage_points)) return rc;
    CK(cudaEventRecord(P.ev[k], P.copy_st));
    CK(cudaStreamWaitEvent(P.comp_st, P.ev[k], 0));
    int rc;
    if (shared_buckets) {
      rc = vt->accumulate(P.ctx, (char*)d_points + off * ab, (char*)P.d_scalars + off * sb, m, k > 0, P.comp_st);
    } else {
      rc = vt->window_sums(P.ctx, (char*)d_points + off * ab, (char*)P.d_scalars + off * sb, m,
                           (char*)P.d_partials + (size_t)k * npart * xb, P.comp_st);
    }
    if (rc) return rc;
    launches += P.ctx->last_launches;
    if (k == fault_after) return set_err(GMSM_ECUDA, "injected fault after batch %d (GMSM_FAULT_AFTER_BATCH)", k);
  }
  if (shared_buckets) {
    P.ctx->last_launches = 0;
    if (int rc = vt->bucket_reduce(P.ctx, P.d_partials, P.comp_st)) return rc;
    launches += P.ctx->last_launches;
    if (h_partials) {
      CK(cudaMemcpyAsync(h_partials, P.d_partials, (size_t)npart * xb, cudaMemcpyDeviceToHost, P.comp_st));
      CK(cudaStreamSynchronize(P.comp_st));
      P.last_launches = launches;
      return GMSM_OK;
    }
    if (int rc = vt->finalize(P.ctx, P.d_partials, 1, P.d_out, P.comp_st)) return rc;
  } else {
    if (int rc = vt->finalize(P.ctx, P.d_partials, nch, P.d_out, P.comp_st)) return rc;
  }
  P.last_launches = launches + 1;
  CK(cudaMemcpyAsync(out_jac, P.d_out, jb, cudaMemcpyDeviceToHost, P.comp_st));
  CK(cudaStreamSynchronize(P.comp_st));
  g_last_oneshot_launches = P.last_launches;
  return GMSM_OK;
}

static int check_device(int device) {
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) return set_err(GMSM_ENODEV, "no CUDA device (%s); this engine has no CPU fallback", cudaGetErrorString(e));
  if (device < 0 || device >= ndev) return set_err(GMSM_EINVAL, "device %d out of range (%d devices)", device, ndev);
  return GMSM_OK;
}

static int check_nb_tasks(int nb_tasks) {
  // (*G1Jac).MultiExp, multiexp.go:67-71
  if (nb_tasks > 1024) return set_err(GMSM_EINVAL, "invalid config: config.NbTasks > 1024");
  return GMSM_OK;
}

// join the W window partials of D shards (host copy, shard-major) on the device of pipeline P0:
// per-window sum over the shards, Horner, normalisation -> out_jac (host)
static int join_partials(int curve, Pipeline& P0, void** d_gather, size_t* gather_cap, const unsigned char* h_part,
                         size_t bytes, int D, uint64_t* out_jac) {
  CurveInfo ci;
  curve_info(curve, &ci);
  CK(cudaSetDevice(P0.device));
  if (*gather_cap < bytes) {
    cudaFree(*d_gather); *d_gather = nullptr;
    CK(cudaMalloc(d_gather, bytes));
    *gather_cap = bytes;
  }
  CK(cudaMemcpyAsync(*d_gather, h_part, bytes, cudaMemcpyHostToDevice, P0.comp_st));
  {
    std::lock_guard<std::mutex> lk2(P0.ctx->mu);
    if (int rc = vtable(curve)->finalize(P0.ctx, *d_gather, D, P0.d_out, P0.comp_st)) return rc;
  }
  CK(cudaMemcpyAsync(out_jac, P0.d_out, 12u * ci.coord_words, cudaMemcpyDeviceToHost, P0.comp_st));
  CK(cudaStreamSynchronize(P0.comp_st));
  return GMSM_OK;
}

// the devices listed in GMSM_DEVICES ("0,1,2,3"), empty if unset
static std::vector<int> env_devices() {
  std::vector<int> out;
  if (const char* e = getenv("GMSM_DEVICES")) {
    for (const char* q = e; *q;) {
      char* end = nullptr;
      long v = strtol(q, &end, 10);
      if (end == q) break;
      out.push_back((int)v);
      q = (*end == ',') ? end + 1 : end;
    }
  }
  return out;
}

// ---- resident bases ----
// device >= 0: all bases on that device.  device == -1: the bases are sharded contiguously over the devices of
// GMSM_DEVICES (one process driving several GPUs); a call then runs one host thread per shard.
struct BaseShard {
  int device = 0;
  size_t lo = 0, hi = 0;
  void* d_points = nullptr;
  Pipeline pipe;
  void* d_gather = nullptr;
  size_t gather_cap = 0;
};
struct gmsm_bases {
  int curve = 0;
  size_t n = 0;
  std::vector<BaseShard> shards;
  std::mutex mu;
};

extern "C" void gmsm_bases_free(gmsm_bases_t* b);

extern "C" gmsm_bases_t* gmsm_bases_upload(gmsm_curve_t curve, const uint64_t* points, size_t n, int device) {
  CurveInfo ci;
  if (!curve_info(curve, &ci)) { set_err(GMSM_EINVAL, "unknown curve id %d", (int)curve); return nullptr; }
  std::vector<int> devs;
  if (device == -1) {
    devs = env_devices();
    if (devs.empty()) { set_err(GMSM_EINVAL, "device = -1 needs GMSM_DEVICES"); return nullptr; }
  } else {
    devs.push_back(device);
  }
  for (int d : devs) if (check_device(d) != GMSM_OK) return nullptr;
  const size_t ab = 8u * ci.coord_words;
  gmsm_bases* b = new gmsm_bases();
  b->curve = curve; b->n = n;
  b->shards.resize(devs.size());
  for (size_t d = 0; d < devs.size(); d++) {
    BaseShard& sh = b->shards[d];
    sh.device = devs[d];
    sh.lo = n * d / devs.size();
    sh.hi = n * (d + 1) / devs.size();
    const size_t bytes = (sh.hi - sh.lo) * ab;
    bool ok = cudaSetDevice(sh.device) == cudaSuccess && cudaMalloc(&sh.d_points, bytes ? bytes : 16) == cudaSuccess;
    if (ok && bytes) ok = cudaMemcpy(sh.d_points, reinterpret_cast<const char*>(points) + sh.lo * ab, bytes, cudaMemcpyHostToDevice) == cudaSuccess;
    if (ok) ok = pipeline_init(sh.pipe, curve, sh.device) == GMSM_OK;
    if (!ok) {
      std::string keep = g_err.empty() ? std::string("upload of bases failed (allocation or H2D copy)") : g_err;
      gmsm_bases_free(b);
      g_err = keep;
      return nullptr;
    }
  }
  return b;
}

// Window tables for resident bases: every shard's point array is replaced by its W-row table (row 0 = the bases,
// row j = 2^(c*j) * bases; W x the memory), built once on the device; later gmsm_bases_multiexp calls run the
// single-bucket-set pass with c ~ 22 (W = 12) instead of c = 17 (W = 15).  Results are bit-identical.
extern "C" int gmsm_bases_precompute(gmsm_bases_t* b, int c) {
  if (!b) return set_err(GMSM_EINVAL, "null bases");
  if (c != 0 && (c < 2 || c > 24)) return set_err(GMSM_EINVAL, "window width c=%d out of range [2,24]", c);
  std::lock_guard<std::mutex> lk(b->mu);
  CurveInfo ci;
  curve_info(b->curve, &ci);
  const size_t ab = 8u * ci.coord_words;
  size_t max_sh = 0;
  for (BaseShard& sh : b->shards) {
    if (sh.pipe.tables) return set_err(GMSM_EINVAL, "window tables already built (c=%d)", sh.pipe.tab_c);
    max_sh = std::max(max_sh, sh.hi - sh.lo);
  }
  if (c == 0) c = choose_c_tables(ci.fr_bits, std::max<size_t>(max_sh, 1));
  const WindowPlan p = make_plan(ci.fr_bits, c);
  if ((double)max_sh * p.nwin >= 2147483000.0)
    return set_err(GMSM_EINVAL, "n*W = %zu*%d does not fit the 31-bit table index; shard the bases", max_sh, p.nwin);
  // build every shard's table first and switch all shards over only when all of them succeeded, so that a
  // failure (typically GMSM_ENOMEM on one device) leaves the handle exactly as it was
  std::vector<void*> tabs(b->shards.size(), nullptr);
  int rc = GMSM_OK;
  for (size_t k = 0; k < b->shards.size() && rc == GMSM_OK; k++) {
    BaseShard& sh = b->shards[k];
    const size_t m = sh.hi - sh.lo;
    const size_t bytes = m * (size_t)p.nwin * ab;
    cudaError_t e = cudaSetDevice(sh.device);
    if (e == cudaSuccess) e = cudaMalloc(&tabs[k], bytes ? bytes : 16);
    if (e != cudaSuccess) {
      cudaGetLastError();   // clear the (non-sticky) allocation error
      rc = set_err(e == cudaErrorMemoryAllocation ? GMSM_ENOMEM : GMSM_ECUDA, "window tables: %zu bytes on device %d: %s", bytes,
                   sh.device, cudaGetErrorString(e));
      break;
    }
    rc = gmsm_tables_build_device((gmsm_curve_t)b->curve, c, sh.d_points, m, tabs[k], m, sh.pipe.comp_st);
    if (rc == GMSM_OK) {
      e = cudaStreamSynchronize(sh.pipe.comp_st);
      if (e != cudaSuccess) rc = set_err(GMSM_ECUDA, "window tables: %s", cudaGetErrorString(e));
    }
  }
  if (rc != GMSM_OK) {
    const std::string keep = g_err;
    for (size_t k = 0; k < tabs.size(); k++)
      if (tabs[k]) { cudaSetDevice(b->shards[k].device); cudaFree(tabs[k]); }
    g_err = keep;
    return rc;
  }
  for (size_t k = 0; k < b->shards.size(); k++) {
    BaseShard& sh = b->shards[k];
    cudaSetDevice(sh.device);
    cudaFree(sh.d_points);
    sh.d_points = tabs[k];
    sh.pipe.tables = true;
    sh.pipe.tab_stride = sh.hi - sh.lo;
    sh.pipe.tab_c = c;
  }
  return GMSM_OK;
}
/* window width / number of table rows of precomputed bases (0 if none) */
extern "C" int gmsm_bases_table_bits(const gmsm_bases_t* b) { return (b && !b->shards.empty() && b->shards[0].pipe.tables) ? b->shards[0].pipe.tab_c : 0; }

extern "C" void gmsm_bases_free(gmsm_bases_t* b) {
  if (!b) return;
  for (BaseShard& sh : b->shards) {
    cudaSetDevice(sh.device);
    pipeline_free(sh.pipe);
    cudaFree(sh.d_points);
    cudaFree(sh.d_gather);
  }
  delete b;
}

extern "C" int gmsm_bases_multiexp(gmsm_bases_t* b, size_t offset, const uint64_t* scalars, size_t n, int nb_tasks,
                                   uint64_t* out_jac) {
  if (!b) return set_err(GMSM_EINVAL, "null bases");
  if (int rc = check_nb_tasks(nb_tasks)) return rc;
  if (offset > b->n || n > b->n - offset) return set_err(GMSM_EINVAL, "len(points) != len(scalars)");
  std::lock_guard<std::mutex> lk(b->mu);
  CurveInfo ci;
  curve_info(b->curve, &ci);
  const size_t ab = 8u * ci.coord_words, xb = 16u * ci.coord_words;
  if (n == 0) { memset(out_jac, 0, 12u * ci.coord_words); return GMSM_OK; }
  // shards intersecting [offset, offset + n)
  struct Job { BaseShard* sh; size_t a, e; };
  std::vector<Job> jobs;
  for (BaseShard& sh : b->shards) {
    const size_t a = std::max(sh.lo, offset), e = std::min(sh.hi, offset + n);
    if (a < e) jobs.push_back({&sh, a, e});
  }
  if (jobs.size() == 1) {
    BaseShard& sh = *jobs[0].sh;
    return pipeline_run(sh.pipe, reinterpret_cast<char*>(sh.d_points) + (jobs[0].a - sh.lo) * ab, nullptr, scalars, n, out_jac);
  }
  // window-table mode: every shard carries the same table width and returns ONE partial
  const bool tables = jobs[0].sh->pipe.tables;
  size_t largest = 0;
  for (const auto& j : jobs) largest = std::max(largest, (size_t)(j.e - j.a));
  // the plan of the largest shard, on all of them
  const int c = tables ? jobs[0].sh->pipe.tab_c : choose_c_for(b->curve, ci.fr_bits, largest, largest_batch(largest, true));
  const WindowPlan plan = make_plan(ci.fr_bits, c);
  const size_t npart = tables ? 1 : (size_t)plan.nwin;
  std::vector<unsigned char> h_part(jobs.size() * npart * xb);
  std::vector<int> rcs(jobs.size(), GMSM_OK);
  std::vector<std::string> errs(jobs.size());
  {
    std::vector<std::thread> th;
    for (size_t k = 0; k < jobs.size(); k++) {
      th.emplace_back([&, k]() {
        const Job& j = jobs[k];
        rcs[k] = pipeline_run(j.sh->pipe, reinterpret_cast<char*>(j.sh->d_points) + (j.a - j.sh->lo) * ab, nullptr,
                              scalars + (j.a - offset) * (size_t)(ci.scalar_bytes / 8), j.e - j.a, nullptr, c, h_part.data() + k * npart * xb);
        if (rcs[k]) errs[k] = g_err;
      });
    }
    for (auto& t : th) t.join();
  }
  for (size_t k = 0; k < jobs.size(); k++)
    if (rcs[k]) return set_err(rcs[k], "device %d: %s", jobs[k].sh->device, errs[k].c_str());
  BaseShard& s0 = *jobs[0].sh;
  return join_partials(b->curve, s0.pipe, &s0.d_gather, &s0.gather_cap, h_part.data(), h_part.size(), (int)jobs.size(), out_jac);
}

// MSM over resident bases with scalars that are ALREADY on the device (the output of a device-side iFFT, gmsm_fft_device:
// prover scalars then never cross PCIe -- SURVEY.md section 8(f) N3).  d_scalars: n x 32 bytes, Montgomery form, on the
// device that holds the bases (single-shard handles only); the work is enqueued on `stream` after whatever the caller put
// there (e.g. the FFT) and the call returns when the result is on the host.
extern "C" int gmsm_bases_multiexp_device(gmsm_bases_t* b, size_t offset, const void* d_scalars, size_t n, int nb_tasks,
                                          uint64_t* out_jac, void* stream) {
  if (!b) return set_err(GMSM_EINVAL, "null bases");
  if (int rc = check_nb_tasks(nb_tasks)) return rc;
  if (offset > b->n || n > b->n - offset) return set_err(GMSM_EINVAL, "len(points) != len(scalars)");
  if (b->shards.size() != 1) return set_err(GMSM_EINVAL, "device scalars need bases that live on one device (this handle is sharded over %zu)", b->shards.size());
  std::lock_guard<std::mutex> lk(b->mu);
  CurveInfo ci;
  curve_info(b->curve, &ci);
  const size_t ab = 8u * ci.coord_words, jb = 12u * ci.coord_words;
  if (n == 0) { memset(out_jac, 0, jb); return GMSM_OK; }
  BaseShard& sh = b->shards[0];
  Pipeline& P = sh.pipe;
  CK(cudaSetDevice(P.device));
  const int c = P.tables ? P.tab_c : choose_c_for(P.curve, ci.fr_bits, n, n);
  if (!P.ctx || P.ctx->max_n < n || P.ctx->max_n > 4 * n + 1024 || P.ctx->plan.c != c || P.ctx->shared != P.tables) {
    if (P.ctx) { gmsm_ctx_destroy(P.ctx); P.ctx = nullptr; }
    P.ctx = ctx_create_ex((gmsm_curve_t)P.curve, n, c, P.device, P.tables);
    if (!P.ctx) return GMSM_ECUDA;
  }
  cudaStream_t st = (cudaStream_t)stream;
  int rc;
  if (P.tables)
    rc = gmsm_ctx_msm_tables_device(P.ctx, sh.d_points, P.tab_stride, offset, d_scalars, n, P.d_out, st);
  else
    rc = gmsm_ctx_msm_device(P.ctx, reinterpret_cast<const char*>(sh.d_points) + offset * ab, d_scalars, n, P.d_out, st);
  if (rc) { cudaStreamSynchronize(st); return rc; }
  CK(cudaMemcpyAsync(out_jac, P.d_out, jb, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return GMSM_OK;
}

// Sessions of the host entry points: device buffers, streams, the pinned ring and the engine context are kept between
// calls (grow-only, shrunk when 4x oversized) so a call costs its copies and kernels, not cudaMalloc.  Each (curve, device)
// pair owns a small POOL of sessions (GMSM_SESSIONS, default 3): a call leases a free one, so concurrent calls -- gnark's
// provers run several MultiExp at once, BenchmarkManyMultiExpG1Reference multiexp_test.go:385-415 -- on different curves,
// different devices or even the same pair proceed in parallel (the H2D of one under the bucket pass of another); a call
// waits only when every session of its pair is taken.  The global mutex guards the table, never a call.
struct Session {
  Pipeline pipe;
  void* d_points = nullptr;
  size_t cap = 0;
  void* d_gather = nullptr;
  size_t gather_cap = 0;
  bool busy = false;
};
static std::mutex g_sess_mu;
static std::condition_variable g_sess_cv;
static std::map<std::pair<int, int>, std::vector<std::unique_ptr<Session>>> g_sessions;

static int session_pool_size() {
  int v = 3;
  if (const char* e = getenv("GMSM_SESSIONS")) v = atoi(e);
  return std::max(1, std::min(v, 16));
}

struct SessionLease {
  Session* S = nullptr;
  SessionLease() = default;
  SessionLease(const SessionLease&) = delete;
  SessionLease& operator=(const SessionLease&) = delete;
  SessionLease(SessionLease&& o) noexcept : S(o.S) { o.S = nullptr; }
  void acquire(int curve, int device) {
    std::unique_lock<std::mutex> lk(g_sess_mu);
    auto& pool = g_sessions[std::make_pair(curve, device)];
    const size_t cap = (size_t)session_pool_size();
    for (;;) {
      for (auto& u : pool) if (!u->busy) { S = u.get(); break; }
      if (!S && pool.size() < cap) { pool.emplace_back(new Session()); S = pool.back().get(); }
      if (S) break;
      g_sess_cv.wait(lk);
    }
    S->busy = true;
  }
  ~SessionLease() {
    if (!S) return;
    { std::lock_guard<std::mutex> lk(g_sess_mu); S->busy = false; }
    g_sess_cv.notify_one();
  }
};

// size the leased session's point buffer for cnt points (exclusive access: the lease)
static int session_prepare(Session& S, int curve, int device, size_t cnt) {
  CurveInfo ci;
  curve_info(curve, &ci);
  CK(cudaSetDevice(device));
  if (int rc = pipeline_init(S.pipe, curve, device)) return rc;
  if (S.cap < cnt || S.cap > 4 * cnt + 1024) {
    cudaFree(S.d_points); S.d_points = nullptr; S.cap = 0;
    CK(cudaMalloc(&S.d_points, cnt * 8u * ci.coord_words));
    S.cap = cnt;
  }
  return GMSM_OK;
}

extern "C" int gmsm_choose_window_bits(gmsm_curve_t curve, size_t n_total) {
  CurveInfo ci;
  if (!curve_info(curve, &ci)) return 0;
  return choose_c_for(curve, ci.fr_bits, n_total, n_total);
}

// one shard of a sharded call, host buffers in, W window partials (host) out: the pipelined engine of
// gmsm_multiexp without the finalize.  All shards must use the same window width c.
extern "C" int gmsm_multiexp_window_sums(gmsm_curve_t curve, const uint64_t* points, const uint64_t* scalars, size_t n, int c,
                                         int device, void* out_partials) {
  CurveInfo ci;
  if (!curve_info(curve, &ci)) return set_err(GMSM_EINVAL, "unknown curve id %d", (int)curve);
  if (c < 2 || c > 24) return set_err(GMSM_EINVAL, "window width c=%d out of range [2,24]", c);
  if (int rc = check_device(device)) return rc;
  const WindowPlan plan = make_plan(ci.fr_bits, c);
  if (n == 0) { memset(out_partials, 0, (size_t)plan.nwin * 16u * ci.coord_words); return GMSM_OK; }
  SessionLease lease;
  lease.acquire(curve, device);
  if (int rc = session_prepare(*lease.S, curve, device, n)) return rc;
  return pipeline_run(lease.S->pipe, lease.S->d_points, points, scalars, n, nullptr, c, out_partials);
}

extern "C" int gmsm_multiexp(gmsm_curve_t curve, const uint64_t* points, const uint64_t* scalars, size_t n, int nb_tasks,
                             uint64_t* out_jac) {
  if (int rc = check_nb_tasks(nb_tasks)) return rc;
  CurveInfo ci;
  if (!curve_info(curve, &ci)) return set_err(GMSM_EINVAL, "unknown curve id %d", (int)curve);
  // devices: GMSM_DEVICES="0,1,2,3" shards one call over several GPUs of this process (one host thread per
  // device, the per-device window partials joined on the first one); default: the single GMSM_DEVICE (0)
  std::vector<int> devs = env_devices();
  if (devs.empty()) {
    int device = 0;
    if (const char* e = getenv("GMSM_DEVICE")) device = atoi(e);
    devs.push_back(device);
  }
  for (int d : devs) if (int rc = check_device(d)) return rc;
  if (n == 0) { memset(out_jac, 0, 12u * ci.coord_words); return GMSM_OK; }
  const size_t ab = 8u * ci.coord_words;
  const size_t D = (n >= ((size_t)1 << 16)) ? devs.size() : 1;   // small calls stay on one device
  if (D == 1) {
    SessionLease lease;
    lease.acquire(curve, devs[0]);
    if (int rc = session_prepare(*lease.S, curve, devs[0], n)) return rc;
    return pipeline_run(lease.S->pipe, lease.S->d_points, points, scalars, n, out_jac);
  }
  // ---- multi-device: contiguous shards (the reference's recursive halving, multiexp.go:128-140) ----
  // one plan for every shard (their partials are added window by window), sized for the work ONE device does: the largest shard
  const size_t shard = (n + D - 1) / D;
  const int c = choose_c_for(curve, ci.fr_bits, shard, largest_batch(shard, false));
  const WindowPlan plan = make_plan(ci.fr_bits, c);
  const size_t xb = 16u * ci.coord_words;
  std::vector<unsigned char> h_part(D * plan.nwin * xb);
  std::vector<int> rcs(D, GMSM_OK);
  std::vector<std::string> errs(D);
  std::vector<SessionLease> leases(D);
  for (size_t d = 0; d < D; d++) {
    const size_t lo = n * d / D, hi = n * (d + 1) / D;
    leases[d].acquire(curve, devs[d]);
    if (int rc = session_prepare(*leases[d].S, curve, devs[d], hi - lo)) return rc;
  }
  {
    std::vector<std::thread> th;
    for (size_t d = 0; d < D; d++) {
      th.emplace_back([&, d]() {
        const size_t lo = n * d / D, hi = n * (d + 1) / D;
        Session& S = *leases[d].S;
        rcs[d] = pipeline_run(S.pipe, S.d_points, points + lo * (ab / 8), scalars + lo * (size_t)(ci.scalar_bytes / 8), hi - lo, nullptr, c,
                              h_part.data() + d * plan.nwin * xb);
        if (rcs[d]) errs[d] = g_err;   // thread-local error text of the worker
      });
    }
    for (auto& t : th) t.join();
  }
  for (size_t d = 0; d < D; d++)
    if (rcs[d]) return set_err(rcs[d], "device %d: %s", devs[d], errs[d].c_str());
  // join on the first device: per-window sum over the D shards, Horner, normalisation
  Session& S0 = *leases[0].S;
  if (int rc = join_partials(curve, S0.pipe, &S0.d_gather, &S0.gather_cap, h_part.data(), h_part.size(), (int)D, out_jac)) return rc;
  int launches = 1;
  for (size_t d = 0; d < D; d++) launches += leases[d].S->pipe.last_launches;
  g_last_oneshot_launches = launches;
  return GMSM_OK;
}

extern "C" int gmsm_bn254_g1_multiexp(const uint64_t* p, const uint64_t* s, size_t n, int t, uint64_t out[12]) { return gmsm_multiexp(GMSM_BN254_G1, p, s, n, t, out); }
extern "C" int gmsm_bn254_g2_multiexp(const uint64_t* p, const uint64_t* s, size_t n, int t, uint64_t out[24]) { return gmsm_multiexp(GMSM_BN254_G2, p, s, n, t, out); }
extern "C" int gmsm_bls12381_g1_multiexp(const uint64_t* p, const uint64_t* s, size_t n, int t, uint64_t out[18]) { return gmsm_multiexp(GMSM_BLS12381_G1, p, s, n, t, out); }
extern "C" int gmsm_bls12381_g2_multiexp(const uint64_t* p, const uint64_t* s, size_t n, int t, uint64_t out[36]) { return gmsm_multiexp(GMSM_BLS12381_G2, p, s, n, t, out); }
extern "C" int gmsm_bls12377_g1_multiexp(const uint64_t* p, const uint64_t* s, size_t n, int t, uint64_t out[18]) { return gmsm_multiexp(GMSM_BLS12377_G1, p, s, n, t, out); }
extern "C" int gmsm_bls12377_g2_multiexp(const uint64_t* p, const uint64_t* s, size_t n, int t, uint64_t out[36]) { return gmsm_multiexp(GMSM_BLS12377_G2, p, s, n, t, out); }
extern "C" int gmsm_secp256k1_g1_multiexp(const uint64_t* p, const uint64_t* s, size_t n, int t, uint64_t out[12]) { return gmsm_multiexp(GMSM_SECP256K1_G1, p, s, n, t, out); }
extern "C" int gmsm_bw6761_g1_multiexp(const uint64_t* p, const uint64_t* s, size_t n, int t, uint64_t out[36]) { return gmsm_multiexp(GMSM_BW6761_G1, p, s, n, t, out); }
extern "C" int gmsm_bw6761_g2_multiexp(const uint64_t* p, const uint64_t* s, size_t n, int t, uint64_t out[36]) { return gmsm_multiexp(GMSM_BW6761_G2, p, s, n, t, out); }
extern "C" int gmsm_bls24315_g1_multiexp(const uint64_t* p, const uint64_t* s, size_t n, int t, uint64_t out[15]) { return gmsm_multiexp(GMSM_BLS24315_G1, p, s, n, t, out); }
extern "C" int gmsm_bls24317_g1_multiexp(const uint64_t* p, const uint64_t* s, size_t n, int t, uint64_t out[15]) { return gmsm_multiexp(GMSM_BLS24317_G1, p, s, n, t, out); }
extern "C" int gmsm_bw6633_g1_multiexp(const uint64_t* p, const uint64_t* s, size_t n, int t, uint64_t out[30]) { return gmsm_multiexp(GMSM_BW6633_G1, p, s, n, t, out); }
extern "C" int gmsm_bw6633_g2_multiexp(const uint64_t* p, const uint64_t* s, size_t n, int t, uint64_t out[30]) { return gmsm_multiexp(GMSM_BW6633_G2, p, s, n, t, out); }

// ------------------------------------------------------------------------------------------
// base generator
// ------------------------------------------------------------------------------------------
extern "C" int gmsm_generate_multiples_device(gmsm_curve_t curve, const uint64_t* base_affine_host, uint64_t start, size_t n,
                                              void* d_out_points, void* stream) {
  CurveInfo ci;
  if (!curve_info(curve, &ci)) return set_err(GMSM_EINVAL, "unknown curve id %d", (int)curve);
  if (n == 0) return GMSM_OK;
  if (int rc = set_device_of(d_out_points)) return rc;
  void* d_base = nullptr;
  const size_t ab = 8u * ci.coord_words;
  CK(cudaMalloc(&d_base, ab));
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaMemcpyAsync(d_base, base_affine_host, ab, cudaMemcpyHostToDevice, st);
  if (e != cudaSuccess) { cudaFree(d_base); return set_err(GMSM_ECUDA, "H2D base: %s", cudaGetErrorString(e)); }
  int rc = vtable(curve)->generate(d_base, start, n, d_out_points, st);
  e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  cudaFree(d_base);
  if (e != cudaSuccess) return set_err(GMSM_ECUDA, "generate_multiples: %s", cudaGetErrorString(e));
  return rc;
}

// ------------------------------------------------------------------------------------------
// N1: fixed-base batch scalar multiplication (host buffers in, host affine points out)
// ------------------------------------------------------------------------------------------
extern "C" int gmsm_batch_scalar_mul(gmsm_curve_t curve, const uint64_t* base_affine, const uint64_t* scalars, size_t n,
                                     uint64_t* out_points) {
  CurveInfo ci;
  if (!curve_info(curve, &ci)) return set_err(GMSM_EINVAL, "unknown curve id %d", (int)curve);
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) return set_err(GMSM_ENODEV, "no CUDA device (%s); this engine has no CPU fallback", cudaGetErrorString(e));
  if (n == 0) return GMSM_OK;
  if (n > 0xFFFFFFF0ull) return set_err(GMSM_EINVAL, "n too large");
  int device = 0;
  if (const char* ev = getenv("GMSM_DEVICE")) device = atoi(ev);
  CK(cudaSetDevice(device));
  // window width: on the GPU the doublings (fr.Bits of them) dominate whatever c is; c = 8 keeps the table
  // (2^7 .. 2^8 points) cache resident.  The result does not depend on c.
  const int c = 8;
  const WindowPlan p = make_plan(ci.fr_bits, c);
  const int maxc = std::max(p.c, p.last_c);
  const size_t tbl = (size_t)1 << (maxc - 1);
  const size_t ab = 8u * ci.coord_words;
  void *d_table = nullptr, *d_scalars = nullptr, *d_out = nullptr;
  cudaStream_t st = nullptr;
  int rc = GMSM_OK;
  auto cleanup = [&]() { cudaFree(d_table); cudaFree(d_scalars); cudaFree(d_out); if (st) cudaStreamDestroy(st); };
  if (cudaMalloc(&d_table, tbl * ab) != cudaSuccess || cudaMalloc(&d_scalars, n * (size_t)ci.scalar_bytes) != cudaSuccess ||
      cudaMalloc(&d_out, n * ab) != cudaSuccess || cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) != cudaSuccess) {
    cleanup();
    return set_err(GMSM_ENOMEM, "gmsm_batch_scalar_mul: device allocation failed");
  }
  rc = gmsm_generate_multiples_device(curve, base_affine, 1, tbl, d_table, st);
  if (rc == GMSM_OK) {
    cudaError_t ce = cudaMemcpyAsync(d_scalars, scalars, n * (size_t)ci.scalar_bytes, cudaMemcpyHostToDevice, st);
    if (ce == cudaSuccess) rc = vtable(curve)->batch_scalar_mul(d_table, d_scalars, n, p.c, p.nwin, d_out, st);
    if (ce == cudaSuccess && rc == GMSM_OK) ce = cudaMemcpyAsync(out_points, d_out, n * ab, cudaMemcpyDeviceToHost, st);
    if (ce == cudaSuccess && rc == GMSM_OK) ce = cudaStreamSynchronize(st);
    if (ce != cudaSuccess) rc = set_err(GMSM_ECUDA, "gmsm_batch_scalar_mul: %s", cudaGetErrorString(ce));
  }
  cleanup();
  return rc;
}

// ------------------------------------------------------------------------------------------
// test hooks
// ------------------------------------------------------------------------------------------
namespace {
struct DevBuf {   // frees on every exit path (the CK macro returns early on errors)
  void* p = nullptr;
  ~DevBuf() { if (p) cudaFree(p); }
  template <class T> T* as() { return reinterpret_cast<T*>(p); }
};
}  // namespace
extern "C" int gmsm_test_op(gmsm_curve_t curve, int op, const uint32_t* a, const uint32_t* b, uint32_t* out, size_t n) {
  int wa = 0, wb = 0, wo = 0;
  const GroupVTable* vt = vtable(curve);
  if (!vt) return set_err(GMSM_EINVAL, "unknown curve id %d", (int)curve);
  vt->test_op_sizes(op, &wa, &wb, &wo);
  if (wo == 0) return set_err(GMSM_EINVAL, "unknown op %d", op);
  if (n == 0) return GMSM_OK;
  DevBuf ba, bb, bo;
  CK(cudaMalloc(&ba.p, n * wa * 4));
  CK(cudaMalloc(&bb.p, n * std::max(wb, 1) * 4));
  CK(cudaMalloc(&bo.p, n * wo * 4));
  uint32_t *da = ba.as<uint32_t>(), *db = bb.as<uint32_t>(), *dout = bo.as<uint32_t>();
  CK(cudaMemcpy(da, a, n * wa * 4, cudaMemcpyHostToDevice));
  if (wb) CK(cudaMemcpy(db, b, n * wb * 4, cudaMemcpyHostToDevice));
  if (int rc = vt->test_op(op, da, db, dout, n)) return rc;
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(out, dout, n * wo * 4, cudaMemcpyDeviceToHost));
  return GMSM_OK;
}

extern "C" int gmsm_test_digits(gmsm_curve_t curve, int c, const uint64_t* scalars, size_t n, uint32_t* out) {
  CurveInfo ci;
  if (!curve_info(curve, &ci)) return set_err(GMSM_EINVAL, "unknown curve id %d", (int)curve);
  if (c < 2 || c > 24) return set_err(GMSM_EINVAL, "c out of range");
  if (n == 0) return GMSM_OK;
  WindowPlan p = make_plan(ci.fr_bits, c);
  DevBuf bs, bo;
  CK(cudaMalloc(&bs.p, n * (size_t)ci.scalar_bytes));
  CK(cudaMalloc(&bo.p, n * (size_t)p.nwin * 4));
  void* ds = bs.p;
  uint32_t* dout = bo.as<uint32_t>();
  CK(cudaMemcpy(ds, scalars, n * (size_t)ci.scalar_bytes, cudaMemcpyHostToDevice));
  if (int rc = vtable(curve)->digits_dump(ds, n, p.c, p.nwin, dout)) return rc;
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(out, dout, n * (size_t)p.nwin * 4, cudaMemcpyDeviceToHost));
  return GMSM_OK;
}

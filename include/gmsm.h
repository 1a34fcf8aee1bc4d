/* gmsm.h -- C ABI of the B200-native multi-scalar-multiplication engine.
 *
 * Drop-in boundary for ConsenSys/gnark-crypto's MultiExp (all citations relative to the
 * reference tree):
 *
 *   (*G1Jac).MultiExp(points []G1Affine, scalars []fr.Element, config ecc.MultiExpConfig)
 *       ecc/bn254/multiexp.go:32        ecc/bls12-381/multiexp.go:32
 *   (*G2Jac).MultiExp                   ecc/bn254/multiexp.go:357       ecc/bls12-381/multiexp.go:355
 *   (*G1Affine).MultiExp / (*G2Affine).MultiExp  (:20, :345) keep calling the Jac version.
 *   ecc.MultiExpConfig{NbTasks int}     ecc/ecc.go:107-110
 *
 * The reference has no FFI; a cgo shim (INTEGRATION.md) binds these symbols from a build-tagged
 * sibling of the generated multiexp.go.  Buffers are passed exactly as Go holds them:
 *
 *   points  : n x {X, Y}; each coordinate L little-endian uint64 limbs in Montgomery form
 *             (L = 4 bn254 / secp256k1, 5 bls24-315 / bls24-317, 6 bls12-381 / bls12-377, 10 bw6-633, 12 bw6-761; G2 coordinates are {A0, A1} pairs, except on
 *             bw6-761 / bw6-633 whose G2 is over Fp); infinity = all zero (g1.go:41-47,178-180).  64 / 96 / 128 / 192 bytes per point.
 *   scalars : n x fr.Limbs uint64 (4; 5 for bw6-633, 6 for bw6-761 -- gmsm_scalar_bytes), Montgomery form, reduced (fr/element.go:36).
 *   out     : Jacobian {X, Y, Z}, 3 x L (G2: 3 x 2L) uint64, Montgomery form.  The engine writes the
 *             affine-normalised representative (X, Y, One), or (0, 0, 0) for infinity.  It is
 *             G1Jac.Equal to what the Go path returns and FromJacobian of it is limb-identical.
 *   Only 8-byte alignment of host pointers is assumed.  All functions are thread-safe.
 *
 * Return value: 0 on success, otherwise a GMSM_E* code; gmsm_last_error() gives the text for the
 * calling thread (the shim turns it into the Go `error`; the two reference error strings,
 * multiexp.go:61-71, are reproduced verbatim).
 */
#ifndef GMSM_H
#define GMSM_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
  GMSM_BN254_G1 = 0,
  GMSM_BN254_G2 = 1,
  GMSM_BLS12381_G1 = 2,
  GMSM_BLS12381_G2 = 3,
  GMSM_BLS12377_G1 = 4,  /* next-row N4: ecc/bls12-377 */
  GMSM_BLS12377_G2 = 5,  /* its Fp2 tower has u^2 = -5 (e2_bls377.go) */
  GMSM_SECP256K1_G1 = 6, /* N4: ecc/secp256k1/multiexp.go:32 -- fp and fr fill all 256 bits */
  GMSM_BW6761_G1 = 7,    /* N4: ecc/bw6-761/multiexp.go:32  -- 12-word Fp, scalars are 6 x uint64 (fr.Bits = 377) */
  GMSM_BW6761_G2 = 8,    /* N4: ecc/bw6-761/multiexp.go:306 -- G2 is also over Fp */
  GMSM_BLS24315_G1 = 9,  /* N4: ecc/bls24-315/multiexp.go:32 -- 5-word Fp (G2 of the bls24 curves is over Fp4: not provided) */
  GMSM_BLS24317_G1 = 10, /* N4: ecc/bls24-317/multiexp.go:32 */
  GMSM_BW6633_G1 = 11,   /* N4: ecc/bw6-633/multiexp.go:32  -- 10-word Fp, scalars are 5 x uint64 (fr.Bits = 315) */
  GMSM_BW6633_G2 = 12    /* N4: ecc/bw6-633/multiexp.go:304 -- G2 over Fp */
} gmsm_curve_t;

enum {
  GMSM_OK = 0,
  GMSM_EINVAL = 1,   /* bad argument (incl. the reference's "invalid config: config.NbTasks > 1024") */
  GMSM_ECUDA = 2,    /* CUDA runtime error */
  GMSM_ENOMEM = 3,   /* device allocation failed */
  GMSM_ENODEV = 4    /* no CUDA device: the engine has NO CPU fallback */
};

const char* gmsm_last_error(void);
const char* gmsm_version(void);

/* sizes in bytes for a curve: affine point, scalar, Jacobian output, one extended-Jacobian partial */
size_t gmsm_affine_bytes(gmsm_curve_t curve);
size_t gmsm_scalar_bytes(gmsm_curve_t curve);
size_t gmsm_jac_bytes(gmsm_curve_t curve);
size_t gmsm_xyzz_bytes(gmsm_curve_t curve);

/* ---- 1. one-shot drop-ins: host buffers in, host Jacobian out (replaces multiexp.go:32 / :357) ----
 * nb_tasks mirrors config.NbTasks: <= 0 means "default", > 1024 is the reference's error; it does
 * not otherwise influence the GPU schedule.  */
int gmsm_bn254_g1_multiexp(const uint64_t* points, const uint64_t* scalars, size_t n, int nb_tasks,
                           uint64_t out_jac[12]);
int gmsm_bn254_g2_multiexp(const uint64_t* points, const uint64_t* scalars, size_t n, int nb_tasks,
                           uint64_t out_jac[24]);
int gmsm_bls12381_g1_multiexp(const uint64_t* points, const uint64_t* scalars, size_t n, int nb_tasks,
                              uint64_t out_jac[18]);
int gmsm_bls12381_g2_multiexp(const uint64_t* points, const uint64_t* scalars, size_t n, int nb_tasks,
                              uint64_t out_jac[36]);
int gmsm_bls12377_g1_multiexp(const uint64_t* points, const uint64_t* scalars, size_t n, int nb_tasks,
                              uint64_t out_jac[18]);   /* ecc/bls12-377/multiexp.go:32 */
int gmsm_bls12377_g2_multiexp(const uint64_t* points, const uint64_t* scalars, size_t n, int nb_tasks,
                              uint64_t out_jac[36]);
int gmsm_secp256k1_g1_multiexp(const uint64_t* points, const uint64_t* scalars, size_t n, int nb_tasks,
                               uint64_t out_jac[12]);  /* ecc/secp256k1/multiexp.go:32 */
int gmsm_bw6761_g1_multiexp(const uint64_t* points, const uint64_t* scalars /* n x 6 */, size_t n, int nb_tasks,
                            uint64_t out_jac[36]);     /* ecc/bw6-761/multiexp.go:32 */
int gmsm_bw6761_g2_multiexp(const uint64_t* points, const uint64_t* scalars /* n x 6 */, size_t n, int nb_tasks,
                            uint64_t out_jac[36]);     /* ecc/bw6-761/multiexp.go:306 (G2 is over Fp as well) */
int gmsm_bls24315_g1_multiexp(const uint64_t* points, const uint64_t* scalars, size_t n, int nb_tasks,
                              uint64_t out_jac[15]);   /* ecc/bls24-315/multiexp.go:32 */
int gmsm_bls24317_g1_multiexp(const uint64_t* points, const uint64_t* scalars, size_t n, int nb_tasks,
                              uint64_t out_jac[15]);   /* ecc/bls24-317/multiexp.go:32 */
int gmsm_bw6633_g1_multiexp(const uint64_t* points, const uint64_t* scalars /* n x 5 */, size_t n, int nb_tasks,
                            uint64_t out_jac[30]);     /* ecc/bw6-633/multiexp.go:32 */
int gmsm_bw6633_g2_multiexp(const uint64_t* points, const uint64_t* scalars /* n x 5 */, size_t n, int nb_tasks,
                            uint64_t out_jac[30]);     /* ecc/bw6-633/multiexp.go:304 */
int gmsm_multiexp(gmsm_curve_t curve, const uint64_t* points, const uint64_t* scalars, size_t n,
                  int nb_tasks, uint64_t* out_jac);
/* sharded calls with one process per GPU: every process runs its shard through the pipelined engine and gets the W
 * window partials back (host memory, W * gmsm_xyzz_bytes); the partials of all shards are then joined with
 * gmsm_ctx_finalize_device.  All shards must pass the same window width (gmsm_choose_window_bits of the TOTAL size).
 * The width returned keeps n_total * W below 2^32 - 296, the context's 32-bit entry limit, whenever some c <= 24 does. */
int gmsm_choose_window_bits(gmsm_curve_t curve, size_t n_total);
int gmsm_multiexp_window_sums(gmsm_curve_t curve, const uint64_t* points, const uint64_t* scalars, size_t n, int c,
                              int device, void* out_partials);
/* kernels launched by the last one-shot call in this process (bench.py's gpu_launches) */
int gmsm_last_oneshot_launches(void);

/* ---- 2. resident bases (the prover flow: SRS / proving-key points are static, kzg.Commit
 * ecc/bn254/kzg/kzg.go:159-176 passes pk.G1[:len(p)]) ---- */
typedef struct gmsm_bases gmsm_bases_t;
/* device >= 0: all bases on that GPU; device == -1: sharded contiguously over the GPUs listed in GMSM_DEVICES
 * (every call then runs one host thread per shard and joins the window partials on the first one) */
gmsm_bases_t* gmsm_bases_upload(gmsm_curve_t curve, const uint64_t* points, size_t n, int device);
/* MSM over bases[offset, offset+n) with host scalars */
int gmsm_bases_multiexp(gmsm_bases_t* bases, size_t offset, const uint64_t* scalars, size_t n,
                        int nb_tasks, uint64_t* out_jac);
void gmsm_bases_free(gmsm_bases_t* bases);
/* the same with scalars that are already in device memory (e.g. the output of gmsm_fft_device: iFFT -> fromMont -> digits
 * without a PCIe crossing, SURVEY.md section 8(f) N3); d_scalars lives on the device of the (single-shard) bases, the work is
 * ordered after `stream`'s earlier work, the result comes back to the host */
int gmsm_bases_multiexp_device(gmsm_bases_t* bases, size_t offset, const void* d_scalars, size_t n, int nb_tasks,
                               uint64_t* out_jac, void* stream);
/* Window tables for resident bases (no reference counterpart: the reference re-reads its bases on every call; this
 * serves the static-SRS flow of kzg.Commit, kzg/kzg.go:159-176).  Replaces the device copy of the bases by a table of
 * W rows, row j = 2^(c*j) * bases (W x the device memory, built once on the GPU).  Afterwards gmsm_bases_multiexp
 * runs ONE bucket set over the n*W table points with the signed digits of partitionScalars (multiexp.go:709-803):
 * no per-window bucket reduction, no Horner (msmReduceChunk), wider windows (c = 22, W = 12 at n = 2^24 instead of
 * c = 17, W = 15).  Results are bit-identical.  c = 0: width from the cost model. */
int gmsm_bases_precompute(gmsm_bases_t* bases, int c);
int gmsm_bases_table_bits(const gmsm_bases_t* bases);   /* c of the tables, 0 if none */

/* ---- 3. device-level engine (device pointers; what bench.py times with inputs resident in HBM and
 * what the multi-GPU path composes).  `stream` is a cudaStream_t (NULL = default stream). ---- */
typedef struct gmsm_ctx gmsm_ctx_t;
/* c = 0: window width from the cost model; otherwise 2 <= c <= 24 (the reference's c in 2..16 are a
 * subset: tests sweep them like multiexp_test.go:95-126) */
gmsm_ctx_t* gmsm_ctx_create(gmsm_curve_t curve, size_t max_n, int c, int device);
void gmsm_ctx_destroy(gmsm_ctx_t* ctx);
int gmsm_ctx_window_bits(const gmsm_ctx_t* ctx);
int gmsm_ctx_num_windows(const gmsm_ctx_t* ctx);
size_t gmsm_ctx_workspace_bytes(const gmsm_ctx_t* ctx);
/* number of kernels launched by the last msm call on this ctx (bench.py's gpu_launches) */
int gmsm_ctx_last_launches(const gmsm_ctx_t* ctx);
/* full MSM: d_out_jac receives the Jacobian triple (device memory, gmsm_jac_bytes) */
int gmsm_ctx_msm_device(gmsm_ctx_t* ctx, const void* d_points, const void* d_scalars, size_t n,
                        void* d_out_jac, void* stream);
/* per-window partial sums only (W extended-Jacobian points, W * gmsm_xyzz_bytes): the per-rank
 * result that ranks exchange over NCCL (reference analogue: the halves joined by AddAssign,
 * multiexp.go:128-140) */
int gmsm_ctx_window_sums_device(gmsm_ctx_t* ctx, const void* d_points, const void* d_scalars, size_t n,
                                void* d_partials, void* stream);
/* combine nranks x W gathered partials: per-window sum over ranks, Horner over windows
 * (msmReduceChunk, multiexp.go:302-315), normalise; d_out_jac as above */
int gmsm_ctx_finalize_device(gmsm_ctx_t* ctx, const void* d_partials, int nranks, void* d_out_jac,
                             void* stream);
/* window-table mode at device level (what gmsm_bases_precompute composes): the context shares one bucket set
 * between all windows; d_table holds gmsm_ctx_num_windows(ctx) rows of row_stride affine points, row j =
 * 2^(c*j) * row 0, built by gmsm_tables_build_device (current device; d_table may alias d_points for row 0).
 * gmsm_ctx_msm_tables_device computes the MSM of scalars[0, n) with the bases row0[offset, offset + n). */
gmsm_ctx_t* gmsm_ctx_create_tables(gmsm_curve_t curve, size_t max_n, int c, int device);
int gmsm_tables_build_device(gmsm_curve_t curve, int c, const void* d_points, size_t n, void* d_table,
                             size_t row_stride, void* stream);
int gmsm_ctx_msm_tables_device(gmsm_ctx_t* ctx, const void* d_table, size_t row_stride, size_t offset,
                               const void* d_scalars, size_t n, void* d_out_jac, void* stream);
/* timings of the last msm call's stages in milliseconds (CUDA events on the call's stream), filled only
 * when enabled with gmsm_ctx_set_profiling(ctx, 1): [digits+hist, scan, scatter, accumulate,
 * carries, bucket-reduce, finalize, total] */
void gmsm_ctx_set_profiling(gmsm_ctx_t* ctx, int on);
int gmsm_ctx_last_stage_ms(gmsm_ctx_t* ctx, float out_ms[8]);

/* ---- 4. base generation (fixed-base helper, SURVEY.md N1/K6): out[i] = [start + i] * base, affine,
 * device pointers; used to build on-curve benchmark inputs without the Go toolchain ---- */
int gmsm_generate_multiples_device(gmsm_curve_t curve, const uint64_t* base_affine_host, uint64_t start,
                                   size_t n, void* d_out_points, void* stream);

/* fixed-base batch scalar multiplication (next-row N1): out[i] = [scalars[i]] * base, affine normal form.
 * Replaces BatchScalarMultiplicationG1 / G2 (ecc/bn254/g1.go:1039-1118, g2.go:1001+), the step before MSM
 * in kzg.NewSRS (kzg/kzg.go:129).  Host buffers; scalars in Montgomery form like everywhere else. */
int gmsm_batch_scalar_mul(gmsm_curve_t curve, const uint64_t* base_affine, const uint64_t* scalars, size_t n,
                          uint64_t* out_points);

/* ---- next-row N2: bulk decoding of serialised G1 points (an SRS in the standard WriteTo format -> resident bases).
 * Replaces G1Affine.SetBytes without the subgroup check -- the Decoder's NoSubgroupChecks path -- ecc/bn254/marshal.go:858-950
 * (:52-60, :952-990), ecc/bls12-381/marshal.go:886-1000: big-endian canonical X (|| Y) with the flag bits of marshal.go:25-31 in
 * the top byte; compressed points take y = (x^3 + b)^((q+1)/4) (fp.Sqrt, q = 3 mod 4) with the sign chosen by
 * LexicographicallyLargest (fp/element.go:282-296).  `bytes` is a homogeneous stream of n points: raw = 1, RawBytes
 * (2 x fp.Bytes each); raw = 0, Bytes (compressed, fp.Bytes each).  check_on_curve != 0 also verifies y^2 = x^3 + b of
 * uncompressed points (for bn254 G1, cofactor 1, that IS the reference's subgroup check).  Output: the reference's in-memory
 * G1Affine (Montgomery limbs, infinity = zeroes).  Errors are the reference's, prefixed by the index of the first bad point.
 * bn254, bls12-381: both forms; bls12-377: raw only (q = 1 mod 4). ---- */
int gmsm_g1_decode(gmsm_curve_t curve, const uint8_t* bytes, size_t n, int raw, int check_on_curve, uint64_t* out_points);
/* device buffers; *d_first_error (8 bytes, device) = (index << 8 | code) of the first bad point, all-ones if none */
int gmsm_g1_decode_device(gmsm_curve_t curve, const void* d_bytes, size_t n, int raw, int check_on_curve, void* d_points,
                          void* d_first_error, void* stream);

/* ---- next-row N3: Fr FFT behind gnark-crypto's fft.Domain (ecc/bn254/fr/fft/domain.go:24-110, fft.go:31-190,
 * bitreverse.go:17-42; ecc/bls12-381/fr/fft identical).  `a` is the []fr.Element image (n x 4 u64, Montgomery),
 * transformed in place; len(a) must equal the domain cardinality.  decimation: GMSM_DIT = 0 (input bit-reversed,
 * output natural), GMSM_DIF = 1 (input natural, output bit-reversed) -- fft.Decimation, fft.go:18-23.  coset != 0
 * = fft.OnCoset().  FFTInverse includes the scaling by CardinalityInv. ---- */
typedef struct gmsm_fft_domain gmsm_fft_domain_t;
enum { GMSM_FR_BN254 = 0, GMSM_FR_BLS12381 = 1, GMSM_FR_BLS12377 = 2 };
enum { GMSM_DIT = 0, GMSM_DIF = 1 };
/* NewDomain(m) / NewDomain(m, WithShift(shift)): cardinality = next power of two >= m; shift = NULL selects
 * GeneratorFullMultiplicativeGroup() (5 / 7), otherwise 4 u64 Montgomery limbs */
gmsm_fft_domain_t* gmsm_fft_domain_create(int fr_field, uint64_t m, const uint64_t* shift, int device);
void gmsm_fft_domain_free(gmsm_fft_domain_t* domain);
uint64_t gmsm_fft_domain_cardinality(const gmsm_fft_domain_t* domain);
/* Generator, GeneratorInv, CardinalityInv, FrMultiplicativeGen, FrMultiplicativeGenInv (5 x 4 u64, Montgomery) */
int gmsm_fft_domain_constants(const gmsm_fft_domain_t* domain, uint64_t out[20]);
int gmsm_fft(gmsm_fft_domain_t* domain, uint64_t* a, size_t n, int decimation, int coset);           /* host buffer */
int gmsm_fft_inverse(gmsm_fft_domain_t* domain, uint64_t* a, size_t n, int decimation, int coset);   /* host buffer */
int gmsm_fft_device(gmsm_fft_domain_t* domain, void* d_a, size_t n, int inverse, int decimation, int coset, void* stream);
int gmsm_fft_bit_reverse_device(gmsm_fft_domain_t* domain, void* d_a, size_t n, void* stream);        /* fft.BitReverse */

/* ---- 5. test hooks: element-wise device functions, used by tests/ to check the sm_100a field and
 * point arithmetic against the oracle.  a, b, out are HOST arrays of n elements each. ---- */
enum {
  GMSM_OP_FMUL = 0, GMSM_OP_FADD = 1, GMSM_OP_FSUB = 2, GMSM_OP_FSQR = 3, GMSM_OP_FNEG = 4,
  GMSM_OP_FDBL = 5, GMSM_OP_FINV = 6,      /* coordinate field (Fp for G1, Fp2 for G2) */
  GMSM_OP_ADD_MIXED = 7,                   /* a: xyzz, b: affine -> xyzz */
  GMSM_OP_SUB_MIXED = 8,
  GMSM_OP_ADD = 9,                         /* a: xyzz, b: xyzz -> xyzz */
  GMSM_OP_DOUBLE = 10,                     /* a: xyzz -> xyzz */
  GMSM_OP_TO_AFFINE = 11,                  /* a: xyzz -> affine */
  GMSM_OP_FR_FROM_MONT = 12,               /* a: scalar -> canonical scalar */
  GMSM_OP_DOT2 = 13,                       /* a: [x | u], b: [y | v] -> x*y + u*v (coordinate field, fused form) */
  GMSM_OP_FP_DOT4 = 14                     /* a: x0..x3, b: y0..y3 -> sum x_k*y_k (base field, fused form) */
};
int gmsm_test_op(gmsm_curve_t curve, int op, const uint32_t* a, const uint32_t* b, uint32_t* out,
                 size_t n);
/* digits of partitionScalars (multiexp.go:709-803) as the device computes them: out[w*n + i] */
int gmsm_test_digits(gmsm_curve_t curve, int c, const uint64_t* scalars, size_t n, uint32_t* out);

#ifdef __cplusplus
}
#endif
#endif /* GMSM_H */

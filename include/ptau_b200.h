/* ptau_b200.h -- C ABI of libptau_b200.so: the B200 (sm_100a) hot path of the
 * Powers-of-Tau -> arkworks KZG preprocessing / loading pipeline.
 *
 * The reference (heliaxdev/kzg-setup-powersoftau) has no FFI layer: its boundary
 * is the crate's pub fns plus three on-disk formats (SURVEY.md 8b).  Each entry
 * point below replaces the per-point loop of one reference function; a Rust
 * caller binds them with `extern "C"` (see INTEGRATION.md and rust/src/ffi.rs).
 *
 *   ptau_convert(ZCASH_UNCOMPRESSED -> ARK_*)   read_g1 / read_g2 loops
 *                                               src/lib.rs:41-54, :56-80, driven by
 *                                               src/bin/preprocess-kgz.rs:140-153,
 *                                               src/bin/preprocess-fastkgz.rs:141-159,
 *                                               src/lib.rs:92-110 (load_phase1)
 *   ptau_convert(ZCASH_COMPRESSED -> ZCASH_UNCOMPRESSED)
 *                                               Accumulator::deserialize(Yes, No) +
 *                                               serialize(No), preprocess-kgz.rs:105-124
 *   ptau_convert(ZCASH_COMPRESSED -> ARK_UNCOMPRESSED)
 *                                               the two above fused (no intermediate file)
 *   ptau_convert(* -> ARK_UNCOMPRESSED)         serialize_uncompressed loops,
 *                                               preprocess-kgz.rs:188-194,
 *                                               preprocess-fastkgz.rs:193-208
 *   ptau_convert(ARK_UNCOMPRESSED -> ARK_MONT_LIMBS)
 *                                               deserialize_unchecked loops,
 *                                               src/lib.rs:179-184, :202-215
 *   ptau_preprocess                             main() of both binaries,
 *                                               preprocess-kgz.rs:162-200,
 *                                               preprocess-fastkgz.rs:180-214
 *   ptau_load_setup                             load_kzg_setup / load_fastkzg_setup,
 *                                               src/lib.rs:174-195, :197-228
 *   ptau_load_phase1                            load_phase1, src/lib.rs:82-121
 *
 * Conventions: all buffers are caller-owned; the library never frees caller
 * memory.  Return value: 0 = ok; > 0 = data error (PTAU_BAD_*), with *bad_index =
 * lowest failing point index of the call (deterministic, independent of the GPU
 * count) and *bad_kind = its PTAU_BAD_* code; < 0 = runtime error (PTAU_ERR_*).
 * One host thread per context.  There is no CPU fallback: every entry point fails
 * with PTAU_ERR_CUDA when no usable sm_100 device is present.
 */
#ifndef PTAU_B200_H
#define PTAU_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default)
#endif

/* groups */
#define PTAU_G1 1
#define PTAU_G2 2

/* point formats */
#define PTAU_FMT_ZCASH_UNCOMPRESSED 1 /* pairing 0.14.2 G{1,2}Uncompressed: BE, 96 / 192 B       */
#define PTAU_FMT_ZCASH_COMPRESSED 2   /* pairing 0.14.2 G{1,2}Compressed:   BE, 48 /  96 B       */
#define PTAU_FMT_ARK_UNCOMPRESSED 3   /* ark-serialize 0.2 serialize_uncompressed: LE, 96 / 192 B */
#define PTAU_FMT_ARK_MONT_LIMBS 4     /* ark-ff 0.2 in-memory Fp384: x,y (G2: c0,c1 each) as      */
                                      /* 6 x u64 Montgomery limbs, then u8 infinity + 7 pad:      */
                                      /* 104 / 200 B                                             */

/* checks bitmask.  Encoding canonicity (coordinates < p, legal flag bits) is
 * always enforced -- the reference has no path that skips it. */
#define PTAU_CHECK_ON_CURVE 2u        /* y^2 = x^3 + 4 (G2: + 4(1+u)); stricter than ark 0.2   */
#define PTAU_CHECK_SUBGROUP 4u        /* same boolean as ark's multiplication by r on EVERY input: */
                                      /* G1 phi(P) = -[z^2]P; G2 psi(P) = [z]P on the twist, and   */
                                      /* the r-multiplication itself for off-curve G2 points       */
#define PTAU_CHECK_REJECT_INFINITY 8u /* point at infinity is an error                          */
/* reference-exact presets */
#define PTAU_CHECKS_LOAD 0u                     /* deserialize_unchecked, src/lib.rs:180        */
#define PTAU_CHECKS_READ PTAU_CHECK_SUBGROUP    /* deserialize_uncompressed, src/lib.rs:52,78   */
#define PTAU_CHECKS_DECOMPRESS 0u               /* CheckForCorrectness::No, preprocess-kgz.rs:108 */
/* default of the drop-in pipeline: everything (identical result on every valid file) */
#define PTAU_CHECKS_STRICT (PTAU_CHECK_ON_CURVE | PTAU_CHECK_SUBGROUP | PTAU_CHECK_REJECT_INFINITY)

/* data errors (> 0) */
#define PTAU_OK 0
#define PTAU_BAD_NON_CANONICAL 1
#define PTAU_BAD_FLAGS 2
#define PTAU_BAD_INFINITY 3
#define PTAU_BAD_NOT_ON_CURVE 4
#define PTAU_BAD_NOT_IN_SUBGROUP 5
#define PTAU_BAD_NOT_POWERS 6 /* ptau_verify_powers: the points are valid but not powers of one tau */
/* runtime errors (< 0) */
#define PTAU_ERR_CUDA (-1)
#define PTAU_ERR_ARG (-2)
#define PTAU_ERR_SIZE (-3)
#define PTAU_ERR_NOMEM (-4)
#define PTAU_ERR_IO (-5)
#define PTAU_ERR_DIGEST (-6) /* BLAKE2b digest of `powersoftau` differs from the expected one */
#define PTAU_ERR_EXISTS (-7) /* `powersoftau_uncompressed` already exists (create_new)       */

/* kzg_setup variants */
#define PTAU_VARIANT_KGZ 1     /* preprocess-kgz / load_kzg_setup         */
#define PTAU_VARIANT_FASTKGZ 2 /* preprocess-fastkgz / load_fastkzg_setup */

typedef struct ptau_ctx ptau_ctx;

typedef struct ptau_timing {
  int n_gpus;
  double wall_ms;      /* host wall clock of the last ptau_convert / pipeline call       */
  double gpu_ms[8];    /* per GPU: first enqueue -> last completion, CUDA events          */
  double kernel_ms[8]; /* per GPU: sum of kernel durations, CUDA events                   */
  uint64_t h2d_bytes[8];
  uint64_t d2h_bytes[8];
  uint64_t kernel_launches; /* kernels launched by the last call, all GPUs              */
} ptau_timing;

/* ---- context ---------------------------------------------------------------- */
int ptau_device_count(void);
/* n_gpus in 1..8; device_ids NULL = 0..n_gpus-1; chunk_points 0 = default (1<<18). */
int ptau_create(ptau_ctx** ctx, int n_gpus, const int* device_ids, size_t chunk_points);
void ptau_destroy(ptau_ctx* ctx);
const char* ptau_strerror(int code);
const char* ptau_last_error(ptau_ctx* ctx); /* CUDA error text of the last PTAU_ERR_CUDA */
int ptau_last_timing(ptau_ctx* ctx, ptau_timing* out);

/* pinned host memory (page-locked, visible to every GPU of the box) */
void* ptau_host_alloc(size_t bytes);
void ptau_host_free(void* p);
int ptau_host_register(void* p, size_t bytes);
int ptau_host_unregister(void* p);

/* ---- layout helpers --------------------------------------------------------- */
size_t ptau_record_size(int group, int fmt);
uint64_t ptau_response_size(uint64_t n_powers);     /* powersoftau CONTRIBUTION_BYTE_SIZE */
uint64_t ptau_uncompressed_size(uint64_t n_powers); /* `powersoftau_uncompressed`         */
uint64_t ptau_setup_size(int variant, uint64_t n_powers); /* `kzg_setup`                  */

/* ---- the per-point path ----------------------------------------------------- */
/* Host buffers in, host buffers out.  Points [0, n_points) are split into
 * contiguous index ranges, one per GPU of the context; each GPU streams its range
 * through double-buffered H2D -> kernel -> D2H and writes its disjoint slice of
 * `out`.  No collective.  `in`/`out` should be pinned for full PCIe speed.  out == NULL
 * validates only: the kernels run, nothing is copied back. */
int ptau_convert(ptau_ctx* ctx, int group, int in_fmt, const void* in, int out_fmt, void* out,
                 size_t n_points, unsigned checks, uint64_t* bad_index, int* bad_kind);

/* Device-resident, asynchronous: one kernel launch on `stream` (a cudaStream_t,
 * NULL = default stream) of the context's GPU slot `gpu`.  d_in / d_out are device
 * pointers, 16-byte aligned.  *d_status is a device u64 the caller sets to
 * PTAU_STATUS_NONE before the first launch; launches fold
 * min((base_index + i) << 8 | kind) over failing points into it. */
#define PTAU_STATUS_NONE 0xffffffffffffffffull
int ptau_convert_device(ptau_ctx* ctx, int gpu, int group, int in_fmt, const void* d_in, int out_fmt,
                        void* d_out, size_t n_points, unsigned checks, uint64_t base_index,
                        uint64_t* d_status, void* stream);
/* returns PTAU_OK or the PTAU_BAD_* kind; fills *bad_index */
int ptau_status_decode(uint64_t status, uint64_t* bad_index);

/* ---- synthetic Powers-of-Tau (known tau) on the GPU -------------------------- */
/* Writes n_points consecutive points [scalar0 * step^(first+i)] * G in `fmt`
 * (ZCASH_COMPRESSED or ZCASH_UNCOMPRESSED) to host memory `out`.  scalars are
 * 32-byte little-endian integers < r.  Used to build synthetic `powersoftau`
 * responses (tau_g1: scalar0 = 1, step = tau; alpha_g1: scalar0 = alpha; ...). */
int ptau_generate(ptau_ctx* ctx, int group, int fmt, const uint8_t scalar0[32], const uint8_t step[32],
                  uint64_t first, size_t n_points, void* out);
int ptau_generate_device(ptau_ctx* ctx, int gpu, int group, int fmt, const uint8_t scalar0[32],
                         const uint8_t step[32], uint64_t first, size_t n_points, void* d_out, void* stream);

/* ---- whole-file pipelines (memory to memory) -------------------------------- */
/* `powersoftau` response (compressed) -> `kzg_setup` bytes; optionally also the
 * `powersoftau_uncompressed` bytes (uncompressed_out may be NULL).  bad_section:
 * 0 tau_g1, 1 tau_g2, 2 alpha_g1, 3 beta_g1, 4 beta_g2. */
int ptau_preprocess(ptau_ctx* ctx, int variant, const void* response, uint64_t response_len,
                    uint64_t n_powers, void* setup_out, uint64_t setup_len, void* uncompressed_out,
                    uint64_t uncompressed_len, unsigned checks, uint64_t* bad_index, int* bad_kind,
                    int* bad_section);
/* same, starting from `powersoftau_uncompressed` bytes (load_powersoftau_accumulator) */
int ptau_preprocess_uncompressed(ptau_ctx* ctx, int variant, const void* uncompressed,
                                 uint64_t uncompressed_len, uint64_t n_powers, void* setup_out,
                                 uint64_t setup_len, unsigned checks, uint64_t* bad_index, int* bad_kind,
                                 int* bad_section);

/* `kzg_setup` bytes -> Montgomery-limb records.  g1_out receives every G1 point of
 * the file in file order (kgz: 2N-1 powers_of_g, N powers_of_gamma_g, g, gamma_g;
 * fastkgz: 2N-1, N), 104 B each; g2_out every G2 point (kgz: h, beta_h; fastkgz: h,
 * beta_h, N powers_of_h), 200 B each.  checks = PTAU_CHECKS_LOAD reproduces the
 * reference; PTAU_CHECKS_STRICT is the validated load. */
int ptau_load_setup(ptau_ctx* ctx, int variant, const void* setup, uint64_t setup_len, uint64_t n_powers,
                    unsigned checks, void* g1_out, uint64_t g1_out_len, void* g2_out, uint64_t g2_out_len,
                    uint64_t* bad_index, int* bad_kind);

/* `phase1radix2m{exp}` bytes -> Montgomery-limb records (alpha, beta_g1, m coeffs_g1,
 * m alpha_coeffs_g1, m beta_coeffs_g1 -> g1_out in that order; beta_g2, m coeffs_g2
 * -> g2_out). */
int ptau_load_phase1(ptau_ctx* ctx, const void* data, uint64_t len, uint64_t m, unsigned checks, void* g1_out,
                     uint64_t g1_out_len, void* g2_out, uint64_t g2_out_len, uint64_t* bad_index,
                     int* bad_kind);

/* ---- file to file (the two binaries' main()) --------------------------------- */
#define PTAU_FILE_SKIP_DIGEST 1u     /* do not check the BLAKE2b digest of `powersoftau`           */
#define PTAU_FILE_NO_UNCOMPRESSED 2u /* fused path: do not write `powersoftau_uncompressed`        */
#define PTAU_FILE_FSYNC 4u           /* fsync the outputs before they are published                */
/* Streams `response_path` through pinned slabs (memory O(slab), not O(N)): size check
 * (preprocess-kgz.rs:83), BLAKE2b-512 digest check against expected_digest_hex (NULL = the
 * ceremony digest of preprocess-kgz.rs:19), `uncompressed_path` created with create_new
 * semantics (:113-118), `setup_path` written in the variant's layout. */
int ptau_preprocess_files(ptau_ctx* ctx, int variant, const char* response_path, const char* setup_path,
                          const char* uncompressed_path, unsigned log2_powers, const char* expected_digest_hex,
                          unsigned flags, unsigned checks, uint64_t* bad_index, int* bad_kind, int* bad_section);
/* load_kzg_setup / load_fastkzg_setup from the file itself (src/lib.rs:174-228), streamed
 * through pinned slabs.  n_powers = 0 infers n from the file size (*n_powers_out receives it).
 * Call once with g1_out = g2_out = NULL and zero lengths to learn n, then with buffers of
 * n_g1*104 and n_g2*200 bytes (kgz: n_g1 = 3n+1, n_g2 = 2; fastkgz: n_g1 = 3n-1, n_g2 = n+2). */
int ptau_load_setup_file(ptau_ctx* ctx, int variant, const char* setup_path, uint64_t n_powers, unsigned checks,
                         void* g1_out, uint64_t g1_out_len, void* g2_out, uint64_t g2_out_len, uint64_t* n_powers_out,
                         uint64_t* bad_index, int* bad_kind);
/* unkeyed BLAKE2b-512 of a file as 128 hex chars + NUL (blake2b_simd, src/lib.rs:128-131) */
int ptau_blake2b_file(const char* path, char out_hex[129]);

/* ---- consumer side (SURVEY 8f-4): KZG10 commit / check --------------------------------- */
/* KZG10 commitment without hiding: commitment = sum_i [coeffs_i] powers_i, the multi-scalar
 * multiplication inside ark-poly-commit 0.2 KZG10::commit (used at src/lib.rs:268-275).
 * powers: n PTAU_FMT_ARK_MONT_LIMBS G1 records (e.g. Powers.powers_of_g from ptau_load_setup);
 * coeffs: n scalars, 32 bytes little-endian each, canonical (< r) and NOT in Montgomery form;
 * commitment: one 104-byte record.  A hiding commitment is commit(p, powers_of_g) +
 * commit(blinding, powers_of_gamma_g): pass both (point, scalar) lists concatenated. */
int ptau_kzg_commit(ptau_ctx* ctx, const void* powers, const void* coeffs, size_t n, void* commitment);

/* Device-resident powers: a setup's powers are the same for every commitment, so they can be uploaded once (a copy
 * on every GPU of the context) and later calls send only the scalars.  ptau_kzg_commit_resident commits to the first
 * n <= n_uploaded powers; same result as ptau_kzg_commit. */
typedef struct ptau_kzg_powers ptau_kzg_powers;
int ptau_kzg_powers_upload(ptau_ctx* ctx, const void* powers, size_t n, ptau_kzg_powers** out);
void ptau_kzg_powers_free(ptau_kzg_powers* powers);
int ptau_kzg_commit_resident(ptau_ctx* ctx, const ptau_kzg_powers* powers, const void* coeffs, size_t n, void* commitment);

/* The polynomial side of KZG10::open (ark-poly-commit 0.2 kzg10 `open` -> `compute_witness_polynomial`, reached from
 * /root/reference/src/lib.rs:276): quotient = (p(X) - p(z)) / (X - z), value = p(z).  coeffs: n scalars (32 bytes LE,
 * < r), quotient_out: (n - 1) scalars, value_out: 32 bytes.  Host arithmetic (a sequential recurrence over Fr); the
 * proof is ptau_kzg_commit(powers, quotient).  No context needed. */
int ptau_kzg_quotient(const void* coeffs, size_t n, const void* point, void* quotient_out, void* value_out);

/* KZG10::open of one polynomial at k points on the GPU (ark-poly-commit 0.2 kzg10 `open` /
 * `compute_witness_polynomial`, reached from src/lib.rs:276).  For each z_j:
 *   values_out[j] = p(z_j),  proofs_out[j] = sum_i q_{j,i} powers_of_g[i],  q_j = (p - p(z_j)) / (X - z_j);
 * with n_b > 0 blinding coefficients also random_v_out[j] = b(z_j) and proofs_out[j] += the same for b over
 * gamma_powers.  powers / gamma_powers: device-resident (ptau_kzg_powers_upload; gamma_powers may be NULL iff n_b = 0).
 * coeffs n, blinding n_b, points k scalars: 32 B LE, < r.  proofs_out k x 104 (ARK_MONT_LIMBS), values_out and
 * random_v_out k x 32 (random_v_out NULL iff n_b = 0).  n > powers' count or n_b > gamma_powers' count
 * (ark: TooManyCoefficients), a non-canonical scalar, or handles of another context: PTAU_ERR_ARG.
 * The quotient is computed on the device (a parallel scan) straight into the MSM's scalars; the points are split in
 * contiguous ranges over the context's GPUs, each opening its points against its own copy of the powers. */
int ptau_kzg_open(ptau_ctx* ctx, const ptau_kzg_powers* powers, const ptau_kzg_powers* gamma_powers,
                  const void* coeffs, size_t n, const void* blinding, size_t n_b, const void* points, size_t k,
                  void* proofs_out, void* values_out, void* random_v_out);

/* KZG10::check for n openings in parallel -- ark-poly-commit 0.2 kzg10 `check`, the call the reference's
 * consumer code makes at /root/reference/src/lib.rs:276-286:
 *     e(C_i - [v_i] g - [rv_i] gamma_g, h) == e(w_i, beta_h - [z_i] h)
 * vk_g1 = {g, gamma_g} (2 x 104-byte ARK_MONT_LIMBS records), vk_g2 = {h, beta_h} (2 x 200 bytes); comms, proofs_w:
 * n x 104; points (z), values (v), random_v: n x 32-byte little-endian scalars < r (random_v may be NULL: proofs
 * without hiding).  ok[i] = 1 when opening i verifies.  Returns PTAU_ERR_ARG for a non-canonical scalar. */
int ptau_kzg_check(ptau_ctx* ctx, const void* vk_g1, const void* vk_g2, const void* comms, const void* points,
                   const void* values, const void* proofs_w, const void* random_v, size_t n, uint8_t* ok);
/* prod_{k<2} e(P_ik, Q_ik) for n items (ark Bls12::product_of_pairings; a pair with a point at infinity counts as 1).
 * g1: n x 2 x 104, g2: n x 2 x 200 (ARK_MONT_LIMBS).  gt_out (may be NULL): n x 576 bytes, the 12 Fq coefficients in
 * arkworks' Fq12 order, canonical little-endian; is_one (may be NULL): n bytes.  KZG10::batch_check is one MSM
 * (ptau_kzg_commit) followed by one such product against {beta_h, h}. */
int ptau_pairing_product2(ptau_ctx* ctx, const void* g1, const void* g2, size_t n, void* gt_out, uint8_t* is_one);

/* ark-ec 0.2 `G2Prepared` of n G2 points (ARK_MONT_LIMBS records): `prepared_h` / `prepared_beta_h` of the keys the
 * reference builds with `h.into()` / `beta_h.into()` (src/lib.rs:223-224, src/bin/preprocess-kgz.rs:177-184).
 * coeffs_out: n x PTAU_G2_PREPARED_COEFFS x 288 bytes -- per coefficient the triple (c0, c1, c2) of Fq2 in ark-ff's
 * in-memory Montgomery limbs, in the order ark pushes them (doubling step, then the addition step on the set bits of
 * |z|); infinity_out[i] = 1 for a point at infinity (ark keeps no coefficients then; the slot is zero-filled). */
#define PTAU_G2_PREPARED_COEFFS 68
int ptau_g2_prepare(ptau_ctx* ctx, const void* g2, size_t n, void* coeffs_out, uint8_t* infinity_out);
/* sum_i [scalars_i] points_i over G2: points = n ARK_MONT_LIMBS G2 records (200 B), scalars 32 B little-endian < r,
 * out: one 200-byte record.  Same conventions, sharding and < r check (PTAU_ERR_ARG) as ptau_kzg_commit. */
int ptau_msm_g2(ptau_ctx* ctx, const void* points, const void* scalars, size_t n, void* out);

/* ---- are the powers powers of one tau? ---------------------------------------------------- */
/* what ptau_verify_powers reads */
#define PTAU_POWERS_RESPONSE 1 /* `powersoftau` response bytes (compressed, ptau_response_size(n) bytes, hash prefix and pubkey included) */
#define PTAU_POWERS_KGZ 2      /* `kzg_setup` of preprocess-kgz     (ptau_setup_size(PTAU_VARIANT_KGZ, n))     */
#define PTAU_POWERS_FASTKGZ 3  /* `kzg_setup` of preprocess-fastkgz (ptau_setup_size(PTAU_VARIANT_FASTKGZ, n)) */
/* relations, reported through *bad_relation (the lowest failing one) */
#define PTAU_REL_GENERATORS 0 /* tau_g1[0] / powers_of_g[0] is the G1 generator, tau_g2[0] / h the G2 generator */
#define PTAU_REL_TAU_G1 1     /* consecutive G1 tau powers have ratio tau (against the first two G2 powers)   */
#define PTAU_REL_TAU_G2 2     /* consecutive G2 tau powers have ratio tau (against the first two G1 powers)   */
#define PTAU_REL_ALPHA_G1 3   /* alpha_tau powers / powers_of_gamma_g have ratio tau                          */
#define PTAU_REL_BETA_G1 4    /* beta_tau powers have ratio tau (response only)                               */
#define PTAU_REL_BETA_G2 5    /* e(beta_g1[0], H) == e(G, beta_g2) (response only)                            */
#define PTAU_REL_KEY 6        /* kgz: g == powers_of_g[0], gamma_g == powers_of_gamma_g[0];                  */
                              /* fastkgz: h == powers_of_h[0], beta_h == powers_of_h[1]                        */
/* Checks that the points of a response or kzg_setup are powers of one tau: tau_g1[i] = [tau^i]G with the G1
 * generator G, alpha powers and beta powers with the same tau, and the G2 powers matching the G1 powers.
 *   Relations checked -- response: GENERATORS, TAU_G1, TAU_G2, ALPHA_G1, BETA_G1, BETA_G2; kgz: GENERATORS, TAU_G1,
 *   ALPHA_G1, KEY (h, beta_h play tau_g2[0], tau_g2[1]); fastkgz: GENERATORS, TAU_G1, TAU_G2, ALPHA_G1, KEY
 *   (powers_of_h[0], powers_of_h[1] play tau_g2[0], tau_g2[1]).
 * Point checks come first: every point is checked with PTAU_CHECKS_STRICT, and a bad point is reported exactly as
 * ptau_preprocess (response: *bad_section, *bad_index within it, *bad_kind) or ptau_load_setup (setups: *bad_index
 * in file order over all points, *bad_section = 0) report the same bytes.  Only when every point is valid are the
 * relations checked; a failure returns PTAU_BAD_NOT_POWERS with the lowest failing relation in *bad_relation.
 * n_powers < 2: PTAU_ERR_ARG; len not the size of the kind for n_powers: PTAU_ERR_SIZE.
 *
 * A ratio relation over a section S of length L with reference pair (Q0, Q1) in G2 holds iff
 *     e(B, Q0) e(-A, Q1) = 1,   A = sum_{i<L-1} rho_{k,i} S_i,   B = sum_{i<L-1} rho_{k,i} S_{i+1}
 * (a G2 section with reference pair (P0, P1) in G1: e(P0, B) e(-P1, A) = 1), where k is the relation number and
 *     rho_{k,i} = BLAKE2b(key = seed, digest 16 bytes)(k as one byte || i as 8 bytes little-endian),
 * read little-endian and cut to its low 127 bits.  Soundness: all points are in the order-r subgroup, so for a seed
 * chosen after the file exists, a file that is not a powers sequence passes a relation with probability at most
 * 2^-127.  A seed known to whoever made the file voids this check.  The check says nothing about whether tau is
 * secret; that is what the ceremony transcript is for.  seed NULL: 32 bytes from getrandom(2).
 *
 * combos_out (may be NULL): 8 slots of 200 bytes; slots 2k-2 and 2k-1 hold A and B of ratio relation k = 1..4 as
 * ARK_MONT_LIMBS records (a G1 record fills the first 104 bytes of its slot); a slot is zero-filled when the relation
 * does not apply to the kind.  Filled only when every point is valid.
 *
 * The file is streamed: device memory per GPU is bounded by the context's chunk_points c (rounded up to a multiple
 * of 16), independent of n_powers -- about 16 c x 540 bytes (at the default c = 2^18: about 2.3 GB) -- so a 2^26
 * response verifies on one GPU. */
int ptau_verify_powers(ptau_ctx* ctx, int kind, const void* data, uint64_t len, uint64_t n_powers,
                       const uint8_t seed[32], uint64_t* bad_index, int* bad_kind, int* bad_section, int* bad_relation,
                       void* combos_out);

/* ---- self-test hook --------------------------------------------------------------- */
/* Raw Fq operations on n pairs of 48-byte Montgomery-limb values (host pointers), computed by
 * the kernels' own field code on the GPU: op 0 mul, 1 add, 2 sub, 3 neg, 4 sqr, 5 a^((p-3)/4),
 * 6 inverse.  Lets tests drive the PTX carry chains with chosen limb patterns. */
int ptau_selftest_fq_op(ptau_ctx* ctx, int gpu, int op, const void* a, const void* b, void* out, size_t n);

/* ---- microbenchmarks used by bench.py for the IMAD roofline denominator ------ */
/* Runs `iters` dependent-chain iterations per thread; returns elapsed ms (CUDA
 * events) in *ms and the number of instructions of the class issued in *ops.
 * kind: 0 = IMAD (32-bit), 1 = IMAD.WIDE.U32.X carry chains, 2 = Fq Montgomery multiplication
 * (ops = multiplications), 3 / 4 = G1 doubling loop with called / inlined multiplications (ops =
 * doublings), 5 = IMAD.WIDE.U32 pure products without carry (measured: half rate, like 1), 6 = DFMA chains,
 * 7 = DFMA chains in the odd warps beside IMAD.WIDE.X rows in the even warps (ops = slots of the shared
 * FMA-heavy pipe: one per DFMA, two per wide MAD). */
int ptau_microbench(ptau_ctx* ctx, int gpu, int kind, int iters, double* ms, double* ops);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* PTAU_B200_H */

/*
 * sipp_b200.h -- C ABI of the B200-native SIPP prover hot path (libsipp_b200.so).
 *
 * This is the drop-in boundary for qope/SIPP's native prover: a Rust host keeps `Transcript`, the arkworks
 * types and the `sipp_prove_native` / `sipp_verify_native` signatures, and calls these entry points where
 * the reference calls into plonky2-bn254-pairing / arkworks (see INTEGRATION.md for the `extern "C"` block).
 * The reference has no FFI of its own; each entry point cites the reference line(s) it replaces.
 *
 * Conventions
 *   - All functions return 0 (SIPP_OK) on success or a negative sipp_status; none of them unwinds.
 *     sipp_last_error() returns a thread-local message for the last failure.
 *   - Byte formats = ark-serialize canonical little-endian integers, uncompressed, WITHOUT flag bits
 *     (`Fq::into_bigint().to_bytes_le()`):
 *        Fq 32 B | Fr 32 B | G1Affine = x||y 64 B | G2Affine = x.c0||x.c1||y.c0||y.c1 128 B
 *        Fq12 = c0.c0.c0, c0.c0.c1, c0.c1.c0, ..., c1.c2.c1 (12 x 32 B = 384 B, arkworks nested order)
 *     The point at infinity is all-zero bytes (ark's `infinity == true` has x = y = 0).
 *   - Host pointers unless a parameter is documented as a device pointer.  The caller owns every buffer.
 *   - One host thread per sipp_ctx; contexts are independent (one per GPU shard / per SIPP instance).
 *   - There is NO CPU fallback: without a CUDA device every compute entry point fails with SIPP_ERR_CUDA.
 */
#ifndef SIPP_B200_H
#define SIPP_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    SIPP_OK = 0,
    SIPP_ERR_CUDA = -1,        /* no device / CUDA runtime failure */
    SIPP_ERR_ARG = -2,         /* bad argument (null pointer, n == 0, n not a power of two where required) */
    SIPP_ERR_LENGTH = -3,      /* A.len() != B.len()          -- reference panics: prover_native.rs:16,27 */
    SIPP_ERR_ZERO_CHALLENGE = -4, /* x.inverse().unwrap()     -- reference panics: prover_native.rs:58 */
    SIPP_ERR_SHORT_PROOF = -5, /* proof.pop().unwrap()        -- reference panics: verifier_native.rs:31,40,42 */
    SIPP_ERR_ENCODING = -6,    /* a field element >= p, a point off the curve or (G2) outside the order-r subgroup */
    SIPP_ERR_VERIFY = -7,      /* Err("Verification failed")  -- verifier_native.rs:83 */
    SIPP_ERR_COMM = -8         /* multi-GPU exchange failed (NCCL missing or in error, host collective callback failed) */
} sipp_status;

typedef struct sipp_ctx sipp_ctx;

/* ---- library ------------------------------------------------------------------------------------------ */
int sipp_init(int device);            /* select the CUDA device of this process (one process per GPU) */
int sipp_shutdown(void);
const char *sipp_last_error(void);
int sipp_device_count(void);          /* 0 when no usable GPU: callers must treat that as fatal */

#define SIPP_OPT_FE_NORMALISATION 1   /* 0 = exact exponent (p^12-1)/r [default, SURVEY A.1 H1], 1 = arkworks multiple */
#define SIPP_OPT_FQ12_ORDER 2         /* transcript order of Fq12: 0 = MyFq12 w-basis [default, SURVEY A.2 H2], 1 = nested */
#define SIPP_OPT_PROFILE 3            /* 1 = record per-kernel CUDA-event timings (sipp_get_stats) */
#define SIPP_OPT_PIPELINE 4           /* 1 = split Miller loop: line kernel + 6-lane cooperative accumulation and final
                                         exponentiation [default]; 0 = one Miller loop per thread (first-round baseline) */
#define SIPP_OPT_WIDE_LINES_MAX 5     /* products of at most this many pairs (summed over the products of a launch) use the
                                         16-lanes-per-pair line kernel (k_lines_wide, latency-bound rounds; also the launches of a batch:
                                         k_lines_wide_batch); 0 = never */
#define SIPP_OPT_FE_ENGINE 6          /* 1 = final exponentiation on the 32-lane Fq12 machine (k_reduce_fe_eng) [default];
                                         0 = 6-lane cooperative version (k_reduce_fe_coop) */
#define SIPP_OPT_WIDE_FOLD_MAX 7      /* folds of at most this many elements per group use the point programs on the lane
                                         engine (k_fold_wide, latency-bound rounds; default 256; a batch uses k_fold_wide_batch up to this + 512 elements); 0 = never */
#define SIPP_OPT_WIDE_ACCUM_MAX 8     /* launches of at most this many pairs accumulate the lines on the 32-lane Fq12 machine
                                         (k_accum_eng) instead of the 6-lane groups of k_accum; 0 = never */
#define SIPP_OPT_BATCH_KPG_MAX 9      /* batched instances: at most this many pairs of one product share an accumulator group */
#define SIPP_OPT_FOLD_STRAUS 10       /* throughput folds: 1 = one thread per element with shared doublings (k_fold_straus) [default];
                                         0 = lane-split components (k_fold_batch / k_fold_split) */
#define SIPP_OPT_BATCH_STREAMS 11     /* batched instances: number of independent sub-batches run on their own streams so that the
                                         latency-bound late rounds overlap (1..8; 0 = default = 1: measured no gain on B200) */
#define SIPP_OPT_BATCH_QLINES 12      /* batched instances: 1 = the line coefficients of every B_i are computed once and shared by Z
                                         and the first Z_L / Z_R (k_qlines_batch + k_eval_lines_batch) [default]; 0 = recomputed */
#define SIPP_OPT_VALIDATE_POINTS 13   /* 1 = every entry point that takes points checks them [default]: A_i on y^2 = x^3 + 3, B_i on the
                                         twist AND in the order-r subgroup (what G1Affine::new / G2Affine::new assert when the reference's
                                         inputs are built); failure = SIPP_ERR_ENCODING.  0 = trusted inputs: the caller guarantees it (the folds
                                         use the GLV / GLS endomorphisms, which act as scalars only on the r-torsion -- results for other points
                                         are unspecified) */
#define SIPP_OPT_MATRIX_TAIL 14       /* single proof: once at most this many points are left (default 32, 0 = off, a power of two <= 64) the prover
                                         computes E[i][j] = e(A_i, B_j) for all pairs and the remaining rounds fold that MATRIX in GT
                                         (E'[i][j] = E[i][j] E[i+h][j+h] E[i+h][j]^x E[i][j+h]^(1/x), k_mat.cu) instead of the points:
                                         same Z_L, Z_R bit for bit, one short kernel per round.  The context's points are then left
                                         as they were when the tail began (only its length keeps halving) */
#define SIPP_OPT_MATRIX_BLOCK_N 15    /* look-ahead stages of the same kind BEFORE the tail: when at most this many points are left (default
                                         256; 0 = off) they are cut into n / 16 blocks, at most SIPP_OPT_MATRIX_BLOCK_R, E[i][j] = <A_block_i, B_block_j> is
                                         computed for all block pairs in one launch set, and log2(R) rounds take Z_L, Z_R from that matrix
                                         while the points are folded on a side stream, off the critical path */
#define SIPP_OPT_MATRIX_FIRST 17      /* 1 [default]: the FIRST stage is built from the inputs themselves (n / 32 blocks, between 8 and 32, inside a budget
                                         of n^2 / 128 (2^9 <= n < 2^12) or 32 n Miller loops, at most 2^18) while the host still hashes A and B: Z is the
                                         product of its diagonal and the first log2(blocks) rounds are one matrix fold each.  10..24 = the
                                         budget is 2^value loops whatever n.  0 = the first rounds run on the points */
#define SIPP_OPT_MATRIX_BLOCK_R 16    /* blocks per look-ahead stage: 4, 8 (default), 16 or 32 (capped so that the stage ends where the tail begins) */
#define SIPP_OPT_PRODUCT_CHUNK_PAIRS 18 /* batched independent products (sipp_inner_product_batch and friends) and the ragged batched prover
                                         (sipp_prove_native_batch_ragged, every round's products) only: at most this many pairs per
                                         line-table chunk; 0 = as many as the 16 GB line-table budget holds [default] */
int sipp_set_option(int option, int value);
int sipp_get_option(int option);

/* ---- prover context: device-resident A, B of the current round ---------------------------------------- */
/* uploads A (n x 64 B) and B (n x 128 B); `let mut A = A.to_vec(); let mut B = B.to_vec();` prover_native.rs:30-31 */
int sipp_ctx_create(const uint8_t *A, const uint8_t *B, size_t n, sipp_ctx **out);
/* same, from DEVICE buffers already in boundary format (no host traffic) */
int sipp_ctx_create_from_device(const void *dA, const void *dB, size_t n, sipp_ctx **out);
int sipp_ctx_destroy(sipp_ctx *ctx);
size_t sipp_ctx_len(const sipp_ctx *ctx);                     /* current n */
/* Z = inner_product(A, B)                                      prover_native.rs:29  (and :15-23) */
int sipp_ctx_inner_product(sipp_ctx *ctx, uint8_t out[384]);
/* Z_L = inner_product(A2, B1), Z_R = inner_product(A1, B2)     prover_native.rs:46-49 */
int sipp_ctx_cross_products(sipp_ctx *ctx, uint8_t zl[384], uint8_t zr[384]);
/* A <- A1 + x A2, B <- B1 + x^-1 B2, n <- n/2                   prover_native.rs:60-74
 * Fold scalars (here and in sipp_gt_fold): little-endian, checked on the host before anything else, in this order: x >= r or
 * x_inv >= r -> SIPP_ERR_ENCODING; x == 0 -> SIPP_ERR_ZERO_CHALLENGE; x x_inv != 1 (mod r) -> SIPP_ERR_ENCODING ("x_inv is not the
 * inverse of x").  A refused fold leaves the context as it was (n, points, stage in progress). */
int sipp_ctx_fold(sipp_ctx *ctx, const uint8_t x[32], const uint8_t x_inv[32]);
/* Opt-in for a host that keeps its own transcript: with stages on, sipp_ctx_inner_product / _cross_products / _fold may run on
 * pairing-matrix stages (SIPP_OPT_MATRIX_*: same Z, Z_L, Z_R bit for bit, several times shorter rounds) exactly as the library's
 * own sipp_prove_native does.  The price: once the tail stage has begun the points are not folded any more, and sipp_ctx_read
 * returns SIPP_ERR_ARG.  Off by default: every call then does literally what its reference line does. */
int sipp_ctx_set_stages(sipp_ctx *ctx, int on);
/* current A, B back to the host (final_A / final_B: verifier_native.rs:74-75; every round in tests) */
int sipp_ctx_read(sipp_ctx *ctx, uint8_t *A_out, uint8_t *B_out);

/* ---- multi-GPU building blocks (for a host that runs its own exchange; the complete prover is below) ---------------- */
/* Writes this shard's un-exponentiated partial products (device format, SIPP_PARTIAL_BYTES each) to DEVICE memory
 * `d_out`, on `stream` (a cudaStream_t; NULL = the legacy default stream, the library orders its own non-blocking
 * stream against it with events): 1 partial for `which` = 0 (Z), 2 for `which` = 1 (Z_L, Z_R).
 * The host all-gathers them (NCCL) and every rank, or rank 0, calls sipp_combine_partials. */
#define SIPP_PARTIAL_BYTES 384
int sipp_ctx_partial_products(sipp_ctx *ctx, int which, void *d_out, void *stream);
/* product over `count` gathered partial sets (layout [rank][nprod][384 B], DEVICE memory), one final exponentiation
 * per product, results to HOST `out` (nprod x 384 B, boundary format) */
int sipp_combine_partials(const void *d_partials, int count, int nprod, uint8_t *out, void *stream);

/* ---- multi-GPU prover inside the library: one process per GPU, strided shards, NCCL on the library stream ---------- */
/* The loop of prover_native.rs:45-75 over `world` ranks.  Rank g holds the pairs i = g (mod world) of A and B
 * ("strided ownership": a pair and its fold partner i + n/2 stay on one rank while n >= 2 world, so folds never move a
 * point).  Per round the reduce kernel writes each rank's two 384-byte partial Miller products into its slot of a gather
 * buffer, ONE in-place ncclAllGather follows on the library stream, rank 0 multiplies the partials, runs one final
 * exponentiation per product, feeds the Fiat-Shamir transcript (which it alone owns: the chain is serial) and broadcasts
 * (x, x^-1); when each rank is down to one pair the `world` pairs are gathered to rank 0, which finishes alone.
 * Call sipp_init(device) first, then ONE of the two sipp_comm_init*; world must be a power of two. */
#define SIPP_COMM_ID_BYTES 128
int sipp_comm_get_unique_id(uint8_t id[SIPP_COMM_ID_BYTES]);   /* rank 0: ncclGetUniqueId; ship the bytes to the other ranks */
int sipp_comm_init(const uint8_t id[SIPP_COMM_ID_BYTES], int rank, int world);   /* ncclCommInitRank on this process's device */
/* the same protocol over the caller's own fabric: collectives on HOST memory (MPI, gloo, a socket ...).  allgather:
 * every rank sends `bytes` from `send`, `recv` receives world x bytes in rank order; broadcast: `buf` of `root` to all.
 * Both return 0 on success.  (Also what the single-GPU tests use to run several ranks on one device.) */
typedef int (*sipp_allgather_fn)(void *user, const void *send, void *recv, size_t bytes);
typedef int (*sipp_broadcast_fn)(void *user, void *buf, size_t bytes, int root);
int sipp_comm_init_host(int rank, int world, sipp_allgather_fn allgather, sipp_broadcast_fn broadcast, void *user);
int sipp_comm_destroy(void);
int sipp_comm_rank(void);
int sipp_comm_world(void);
int sipp_comm_nccl_version(void);     /* ncclGetVersion of the libnccl bound at run time (dlopen), 0 if there is none */
/* pub fn sipp_prove_native(A, B) -> Vec<Fq12>   prover_native.rs:26-80, collectively: every rank passes its strided shard
 * (n / world pairs: A_local[j] = A[j * world + rank]) and the TOTAL n; rank 0 also passes the full A, B (the transcript
 * absorbs every input point, :36-39) and receives the proof ((2 log2 n + 1) x 384 B, returned order); the other ranks may
 * pass NULL for A_full, B_full and proof.  Without a communicator this is sipp_prove_native on one GPU.
 * Folds stay local (index i and its partner i + n/2 share a rank) until the tail moves to rank 0 -- by default where rank 0's
 * look-ahead stages begin (SIPP_OPT_MATRIX_BLOCK_N points left, 256), at the latest at one pair per rank. */
int sipp_prove_native_sharded(const uint8_t *A_local, const uint8_t *B_local, size_t n, const uint8_t *A_full, const uint8_t *B_full,
                              uint8_t *proof);
/* same with the shard already resident in HBM (DEVICE pointers, boundary format) */
int sipp_prove_native_sharded_device(const void *dA_local, const void *dB_local, size_t n, const uint8_t *A_full, const uint8_t *B_full,
                                     uint8_t *proof);
/* The protocol loop itself with the compute / exchange side supplied by the caller (the library's own backend is the
 * CUDA kernels + the communicator above).  Host code only: it needs no GPU, which is how the CPU tests run the loop.
 * products(which): this rank's partial products of the round (0: Z; 1: Z_L, Z_R) and their all-gather; combine: rank 0,
 * product over the ranks + one final exponentiation per product -> nprod x 384 B; broadcast: SIPP_SHARD_XS_BYTES from
 * rank 0 (x || x^-1 || status); fold: A <- A1 + x A2, B <- B1 + x^-1 B2 on the local shard; collapse: gather the last pair
 * of every rank to rank 0, after which rank 0's products / combine are local.  All return 0 or a negative sipp_status. */
#define SIPP_SHARD_XS_BYTES 72
typedef struct sipp_shard_backend {
    void *user;
    int rank, world;
    size_t (*local_len)(void *user);
    int (*products)(void *user, int which);
    int (*combine)(void *user, int nprod, uint8_t *out);
    int (*broadcast)(void *user, uint8_t *xs);
    int (*fold)(void *user, const uint8_t *x, const uint8_t *x_inv);
    int (*collapse)(void *user);
} sipp_shard_backend;
int sipp_prove_native_sharded_backend(const sipp_shard_backend *backend, size_t n, const uint8_t *A_full, const uint8_t *B_full,
                                      uint8_t *proof);

/* ---- stand-alone operations --------------------------------------------------------------------------- */
/* pairing(a, b)                                                verifier_native.rs:80, prover_native.rs:20 */
int sipp_pairing(const uint8_t a[64], const uint8_t b[128], uint8_t out[384]);
/* pub fn inner_product(A, B) -> Fq12                           prover_native.rs:15 */
int sipp_inner_product(const uint8_t *A, const uint8_t *B, size_t n, uint8_t out[384]);
/* x.inverse() in Fr                                            prover_native.rs:58 */
int sipp_fr_inverse(const uint8_t x[32], uint8_t out[32]);
/* Z_L.pow(x) * Z * Z_R.pow(inv_x)                              verifier_native.rs:59-61
 * x, x_inv: the fold-scalar checks of sipp_ctx_fold, made before the device is touched */
int sipp_gt_fold(const uint8_t zl[384], const uint8_t z[384], const uint8_t zr[384], const uint8_t x[32],
                 const uint8_t x_inv[32], uint8_t out[384]);

/* ---- batched independent products: many inner products of unequal lengths (and many pairings) in one call ---------------- */
/* count independent products, CSR segments: out[j] = prod_{offsets[j] <= i < offsets[j+1]} e(A_i, B_i)  (inner_product,
 * prover_native.rs:15-23, per segment).  offsets: count + 1 HOST entries, offsets[0] = 0, non-decreasing, offsets[count] = a_len.
 * An empty segment gives Fq12::one().  out: count x 384 B, boundary format.  Points validated as for sipp_inner_product.
 * Every out[j] is byte-identical to sipp_inner_product on its segment (GT products are exact: the grouping of the multiplications
 * does not change the bits), under either SIPP_OPT_FE_NORMALISATION.
 *   - a_len != b_len: SIPP_ERR_LENGTH; a NULL pointer (count > 0) or bad offsets: SIPP_ERR_ARG -- both before the device is touched.
 *   - count == 0: returns what sipp_init(0) would (SIPP_ERR_CUDA without a device) and writes nothing.
 *   - a coordinate >= p, or with SIPP_OPT_VALIDATE_POINTS a point off the curve or a G2 point outside the subgroup, fails the whole
 *     call with SIPP_ERR_ENCODING and writes nothing.  Identity points (all-zero bytes) contribute the factor 1.
 *   - Always the split pipeline (lines + 6-lane accumulation); SIPP_OPT_PIPELINE is not read.  SIPP_OPT_FE_ENGINE,
 *     SIPP_OPT_WIDE_LINES_MAX, SIPP_OPT_BATCH_KPG_MAX (pairs per accumulator group, at most) and SIPP_OPT_PRODUCT_CHUNK_PAIRS apply.
 *   - sipp_stats.miller_pairs grows by a_len. */
int sipp_inner_product_batch(const uint8_t *A, size_t a_len, const uint8_t *B, size_t b_len, const size_t *offsets, size_t count,
                             uint8_t *out);
/* same, A / B / out in DEVICE memory (boundary format); offsets stay on the host */
int sipp_inner_product_batch_device(const void *dA, const void *dB, size_t n, const size_t *offsets, size_t count, void *d_out);
/* out[j] = pairing(a_j, b_j)  (verifier_native.rs:80) for j < count: the batch above with one pair per segment */
int sipp_pairing_batch(const uint8_t *a, const uint8_t *b, size_t count, uint8_t *out);

/* ---- batched multi-scalar multiplications: many independent MSMs of unequal lengths in G1 and G2 in one call ----------------- */
/* count independent MSMs, CSR segments: out[j] = sum_{offsets[j] <= i < offsets[j+1]} [k_i] P_i.
 *   - Formats: points in the boundary format (G1 64 B, G2 128 B; the identity is all-zero bytes), scalars 32 B little-endian integers,
 *     one per point.  out: count x 64 B (G1) or count x 128 B (G2) canonical affine points; an empty segment, or a sum that is the
 *     identity, gives all-zero bytes.  The results are canonical group elements: every out[j] is byte-identical to the sum of the
 *     [k_i] P_i of its segment computed any other way.
 *   - offsets: count + 1 HOST entries, offsets[0] = 0, non-decreasing, offsets[count] = n (as sipp_inner_product_batch).
 *     count == 0 with n == 0 returns what sipp_init(0) would (SIPP_ERR_CUDA without a device) and writes nothing.
 *   - SIPP_ERR_ARG: a NULL pointer (count > 0), bad offsets, count == 0 with n > 0, or n > 2^32 - 1; all before the device is touched.
 *     Valid arguments without a device give SIPP_ERR_CUDA.
 *   - Host forms: a scalar >= r, then a coordinate >= p, is refused on the host with SIPP_ERR_ENCODING before the device is touched.
 *     Device forms: the same checks run on the device; a failure fails the whole call with SIPP_ERR_ENCODING and nothing is written
 *     to d_out.  Both forms report the first failure in this order: a scalar >= r, a coordinate >= p, a point off the curve, a G2
 *     point outside the subgroup (sipp_last_error names it).  With SIPP_OPT_VALIDATE_POINTS = 1 (default) a point off the curve, or a G2 point outside the order-r subgroup, is
 *     refused the same way; with 0 the caller guarantees the points, and results for points outside the r-torsion are unspecified
 *     (the kernels use the GLV / GLS endomorphisms, which act as scalars only there).
 *   - Path per segment, chosen from its length alone (sipp_test_msm_plan shows it): fewer than 13 (G1) or 8 (G2) points, Straus (one thread per
 *     segment, doublings shared by the 2 (G1) or 4 (G2) GLV / GLS sub-scalars of all its points); from there on, Pippenger with
 *     signed c-bit windows, c from 5 to 16 growing with the length.
 *   - Device scratch, returned to the library's pool on return, per point: NC W sort entries of 16 B (keys and values, double-buffered
 *     for the sort) with their chunk partials (12 B per entry in G1, 24 B in G2), NC terms (64 B G1, 128 B G2) and, when its segment
 *     takes the Straus path, NC x 44 B of NAF digits; NC = 2 (G1) or 4 (G2), W = 128 / c + 1 (G1) or 66 / c + 1 (G2) windows, at most
 *     26 / 14 -- about 2.1 KB per G1 point and 3.4 KB per G2 point at most -- plus W 2^(c-1) Jacobian buckets (96 B G1, 192 B G2) per
 *     Pippenger segment and the sort's own scratch.  More than 2^31 terms, sort entries or buckets, or more than 2^32 - 1 segments,
 *     give SIPP_ERR_CUDA; calls of 2^20 points per group are supported.
 *   - The device forms: points, scalars and d_out in DEVICE memory (4-byte aligned); offsets stay on the host.  Before reading any
 *     input the library stream waits for the legacy default stream, so inputs just written there need no synchronisation; the call
 *     returns once d_out is complete.  No option other than SIPP_OPT_VALIDATE_POINTS is read; sipp_stats.launches grows, no other
 *     counter changes. */
int sipp_g1_msm_batch(const uint8_t *points, const uint8_t *scalars, size_t n, const size_t *offsets, size_t count, uint8_t *out);
int sipp_g2_msm_batch(const uint8_t *points, const uint8_t *scalars, size_t n, const size_t *offsets, size_t count, uint8_t *out);
int sipp_g1_msm_batch_device(const void *d_points, const void *d_scalars, size_t n, const size_t *offsets, size_t count, void *d_out);
int sipp_g2_msm_batch_device(const void *d_points, const void *d_scalars, size_t n, const size_t *offsets, size_t count, void *d_out);

/* ---- batched multi-exponentiations in GT (Fq12): many independent products of powers of unequal lengths in one call --------------- */
/* count independent multi-exponentiations, CSR segments: out[j] = prod_{offsets[j] <= i < offsets[j+1]} g_i^(k_i), computed in Fq12 as a
 * field, exactly as the reference's `Z_L.pow(x)` (square-and-multiply over the bits of the integer) followed by products.  Products in
 * Fq12 are exact, so every out[j] is byte-identical to that computation for EVERY Fq12 input: elements outside GT, non-units and zero
 * (0^0 = 1, 0^k = 0 for k >= 1) included.  No GT membership is assumed or checked.
 *   - Formats: elements in the boundary format (Fq12, 384 B, arkworks nested order), scalars 32 B little-endian integers, one per element.
 *     out: count x 384 B; an empty segment gives Fq12::one().
 *   - offsets: count + 1 HOST entries, offsets[0] = 0, non-decreasing, offsets[count] = n (as sipp_inner_product_batch).
 *     count == 0 with n == 0 returns what sipp_init(0) would (SIPP_ERR_CUDA without a device) and writes nothing.
 *   - SIPP_ERR_ARG: a NULL pointer (count > 0), bad offsets, count == 0 with n > 0, or n > 2^32 - 1; all before the device is touched.
 *     Valid arguments without a device give SIPP_ERR_CUDA.
 *   - Host form: a scalar >= r, then a coordinate >= p, is refused on the host with SIPP_ERR_ENCODING before the device is touched.
 *     Device form: the same checks run on the device; a failure fails the whole call with SIPP_ERR_ENCODING and nothing is written to
 *     d_out.  Both forms report the first failure in this order: a scalar >= r, then a coordinate >= p (sipp_last_error names it).
 *   - Path per segment, chosen from its length alone (sipp_test_gt_msm_plan shows it): fewer than 512 elements, one generic power per
 *     element (6 lanes each) and a segmented product; from there on, Pippenger with unsigned c-bit windows (ceil(254 / c) windows of
 *     2^c - 1 buckets), c from 2 to 16 growing with the length.  No Frobenius split, cyclotomic squaring or inverse is used.
 *   - Device scratch, returned to the library's pool on return, per element: 384 B (decoded table) and, on the short path, 32 B; on the
 *     Pippenger path W sort entries of 16 B (keys and values, double-buffered for the sort) with 48 B of chunk partials each, W =
 *     ceil(254 / c) (at most 127; 16 at 2^20 elements); per Pippenger segment W (2^c - 1) buckets and W ceil((2^c - 1) / 512) window
 *     partials of 384 B (about 400 MB for one segment of 2^20 elements); plus the sort's own scratch.  More than 2^31 - 1 elements, sort
 *     entries or buckets, more than 2^32 - 1 segments, or scratch the device cannot hold, give SIPP_ERR_CUDA with a message and write
 *     nothing; calls of 2^20 elements are supported.
 *   - The device form: elements, scalars and d_out in DEVICE memory (4-byte aligned; inputs are read one word at a time); offsets stay on
 *     the host.  Before reading any input the library stream waits for the legacy default stream, so inputs just written there need no
 *     synchronisation; the call returns once d_out is complete; copies use cudaMemcpyAsync.
 *   - No option is read (SIPP_OPT_VALIDATE_POINTS included: there are no points, and the encoding checks always run; no pairing or
 *     transcript is involved, so the H1 / H2 switches do not apply).  sipp_stats.launches grows, no other counter changes. */
int sipp_gt_msm_batch(const uint8_t *elems, const uint8_t *scalars, size_t n, const size_t *offsets, size_t count, uint8_t *out);
int sipp_gt_msm_batch_device(const void *d_elems, const void *d_scalars, size_t n, const size_t *offsets, size_t count, void *d_out);

/* ---- Fiat-Shamir transcript (host; Poseidon over Goldilocks)  transcript_native.rs:14-66 ---------------- */
typedef struct { uint64_t state[4]; } sipp_transcript;
void sipp_transcript_new(sipp_transcript *t);                                          /* :19-23 */
void sipp_transcript_append(sipp_transcript *t, const uint64_t *msg, size_t n);        /* :25-30 */
void sipp_transcript_append_fq12(sipp_transcript *t, const uint8_t f[384]);            /* :32-40 */
void sipp_transcript_append_g1(sipp_transcript *t, const uint8_t a[64]);               /* :42-46 */
void sipp_transcript_append_g2(sipp_transcript *t, const uint8_t b[128]);              /* :48-54 */
void sipp_transcript_get_challenge(const sipp_transcript *t, uint8_t x[32]);           /* :56-65 */
/* absorb n (A_i, B_i) pairs in order: the loop at prover_native.rs:36-39 / verifier_native.rs:25-28 */
void sipp_transcript_append_pairs(sipp_transcript *t, const uint8_t *A, const uint8_t *B, size_t n);
void sipp_poseidon_permute(uint64_t state[12]);          /* AVX-512 when the CPU has it, else portable */
void sipp_poseidon_permute_portable(uint64_t state[12]);
int sipp_poseidon_backend(void);                          /* 2 = AVX-512 IFMA, 1 = AVX-512, 0 = portable (SIPP_POSEIDON=avx512|portable forces a slower one) */
double sipp_poseidon_ns_per_permutation(long count);      /* measured on this CPU: a dependent chain of `count` permutations, best of three */

/* ---- whole protocol with the C++ host transcript inside (what the Python mirror and bench.py call) ------ */
/* pub fn sipp_prove_native(A, B) -> Vec<Fq12>                  prover_native.rs:26-80
 * proof: (2 log2 n + 1) x 384 B in the returned (reversed) order [Z_R(last), Z_L(last), ..., Z_R(1), Z_L(1), Z] */
int sipp_prove_native(const uint8_t *A, size_t a_len, const uint8_t *B, size_t b_len, uint8_t *proof);
size_t sipp_proof_len(size_t n);      /* number of Fq12 elements = 2 log2 n + 1 */
/* same protocol on an existing context (inputs already resident in HBM); A/B host copies feed the transcript */
int sipp_ctx_prove(sipp_ctx *ctx, const uint8_t *A, const uint8_t *B, uint8_t *proof);
/* pub fn sipp_verify_native(A, B, proof) -> Result<SIPPStatement>   verifier_native.rs:14-85
 * returns SIPP_OK for Ok(statement), SIPP_ERR_VERIFY for Err; the statement's computed members are written to
 * final_A[64], final_B[128], final_Z[384] when non-NULL (A, B, Z are the caller's own inputs: statements.rs:80-88) */
int sipp_verify_native(const uint8_t *A, size_t a_len, const uint8_t *B, size_t b_len, const uint8_t *proof, size_t proof_len,
                       uint8_t *final_A, uint8_t *final_B, uint8_t *final_Z);
/* Proof and statement in one call: sipp_prove_native, plus the statement members that sipp_verify_native would write for
 * (A, B, proof) -- final_A[64], final_B[128], final_Z[384], byte-identical -- without a verification pass.  The proof bytes are those
 * of sipp_prove_native.  final_A / final_B are the points folded down to one (verifier_native.rs:74-75) and final_Z, which the
 * verifier computes as Z prod Z_L^x Z_R^(1/x) (:59-61), is pairing(final_A, final_B) by bilinearity: the output satisfies
 * pairing(final_A, final_B) == final_Z by construction, under either SIPP_OPT_FE_NORMALISATION, so the call returns SIPP_OK
 * exactly where sipp_verify_native on its proof returns Ok(statement).  The statement's A, B and Z are the caller's inputs and the
 * proof's last element.
 *   - Each of final_A, final_B, final_Z may be NULL; that member is then not written (nor computed where skipping is free).
 *   - Argument checks, their order and codes are those of sipp_prove_native, all before the device is touched; valid arguments
 *     without a device give SIPP_ERR_CUDA.  A bad point (SIPP_ERR_ENCODING) or a zero challenge (SIPP_ERR_ZERO_CHALLENGE) fails the
 *     call, and then nothing is written to `proof` or to any final buffer.
 *   - Options: those of sipp_prove_native; every value gives the same bytes.  With a pairing-matrix tail stage (the defaults) the
 *     tail keeps folding the points on the side stream and final_Z is its 1 x 1 matrix after the last round; without one
 *     (SIPP_OPT_MATRIX_TAIL = 0, SIPP_OPT_PIPELINE = 0 or SIPP_OPT_FE_ENGINE = 0) final_Z is one pairing of the folded points.
 *     n = 1: final_A = A, final_B = B, final_Z = Z.
 *   - sipp_stats: miller_pairs and fold_points grow exactly as for sipp_prove_native, plus miller_pairs by 1 when n >= 2, final_Z
 *     is non-NULL and no tail stage ran (the pairing of the folded points).  launches grows by more than for sipp_prove_native
 *     (the tail's point folds, the last matrix fold and its encode, the encodes of final_A and final_B); that count is not part of
 *     the contract. */
int sipp_prove_native_statement(const uint8_t *A, size_t a_len, const uint8_t *B, size_t b_len, uint8_t *proof,
                                uint8_t *final_A, uint8_t *final_B, uint8_t *final_Z);

/* ---- witness hand-off to the untouched circuit side (host only, no GPU) --------------------------------------------------- */
/* The u32 public-input vector of a SIPPStatement: what `SIPPStatement::from_vec` parses (statements.rs:133-170) and the verifier
 * circuit emits (`SIPPStatementTarget::to_vec`, statements.rs:24-39; compared at verifier_circuit.rs:255-268).  8 little-endian
 * limbs per Fq: A (n x 16) | B (n x 32) | Z (96) | final_A (16) | final_B (32) | final_Z (96); an Fq12 is `MyFq12.coeffs`
 * (statements.rs:120-131; order switch SIPP_OPT_FQ12_ORDER as for the transcript). */
size_t sipp_statement_u32_len(size_t n);                 /* 48 n + 240 */
int sipp_statement_to_u32(const uint8_t *A, const uint8_t *B, size_t n, const uint8_t Z[384], const uint8_t final_A[64],
                          const uint8_t final_B[128], const uint8_t final_Z[384], uint32_t *out, size_t out_len);
/* SIPP_ERR_LENGTH when in_len != sipp_statement_u32_len(n) (the reference asserts, statements.rs:139); SIPP_ERR_ENCODING for a
 * limb group >= p */
int sipp_statement_from_u32(size_t n, const uint32_t *in, size_t in_len, uint8_t *A, uint8_t *B, uint8_t Z[384], uint8_t final_A[64],
                            uint8_t final_B[128], uint8_t final_Z[384]);

/* ---- batched instances: `count` independent proofs in lock-step (BASELINE config "4096 independent n=128 instances") ---- */
/* Equivalent to `count` calls of sipp_prove_native (prover_native.rs:26-80) on A[j*n .. (j+1)*n), B[j*n .. (j+1)*n):
 * proofs = count x sipp_proof_len(n) x 384 B, instance j's proof at proofs + j * sipp_proof_len(n) * 384 in the returned
 * (reversed) order.  Round k of every instance runs in the same launches; each instance keeps its own Fiat-Shamir chain
 * (transcript_native.rs:14-66) ON THE DEVICE, so nothing crosses PCIe between the upload and the proofs.  Instances are
 * independent: a multi-GPU host gives each rank its own slice of instances, no collective. */
int sipp_prove_native_batch(const uint8_t *A, const uint8_t *B, size_t n, size_t count, uint8_t *proofs);
/* `count` verifications in lock-step (verifier_native.rs:14-85 per instance): results[j] = SIPP_OK for Ok(statement),
 * SIPP_ERR_VERIFY for Err("Verification failed"), SIPP_ERR_ENCODING for a proof with a coordinate >= p; every instance's proof is proof_len x 384 B (>= sipp_proof_len(n), read
 * from its end like the reference's pop()).  final_A (count x 64 B), final_B (count x 128 B), final_Z (count x 384 B) receive
 * the computed statement members when non-NULL.  The return value reports whether the batch ran, not whether proofs verified. */
int sipp_verify_native_batch(const uint8_t *A, const uint8_t *B, size_t n, size_t count, const uint8_t *proofs, size_t proof_len,
                             int *results, uint8_t *final_A, uint8_t *final_B, uint8_t *final_Z);
/* sipp_verify_native_batch with every buffer in DEVICE memory (boundary format, 4-byte aligned): dA, dB, d_proofs as for the host form,
 * d_results count x int32, d_final_A / _B / _Z count x 64 / 128 / 384 B, each final may be NULL.  results[j] and every final are
 * byte-identical to the host form's on the same bytes and options: the finals are written for every instance, SIPP_ERR_ENCODING ones
 * included.  A, B and the proofs are only read, in place; no input crosses PCIe.
 *   - Argument checks, all before the device is touched: a NULL dA, dB or d_proofs, count == 0, n not a non-zero power of two, then
 *     a NULL d_results: SIPP_ERR_ARG; then proof_len < sipp_proof_len(n): SIPP_ERR_SHORT_PROOF.  Valid arguments without a device give
 *     SIPP_ERR_CUDA.  One difference: sipp_verify_native_batch initialises the device first, so without a device it returns
 *     SIPP_ERR_CUDA for bad arguments too, where this call returns their own codes.
 *   - A bad point or a zero challenge fails the whole call, and then nothing is written to d_results or the finals.
 *   - The library stream waits for the work already enqueued on the legacy default stream (torch's current stream unless the caller
 *     switched streams) before it reads an input; the call returns when the results and finals are complete.
 *   - Options and sipp_stats.fold_points / miller_pairs as for the host form; launches grows by more (not part of the contract). */
int sipp_verify_native_batch_device(const void *dA, const void *dB, size_t n, size_t count, const void *d_proofs, size_t proof_len,
                                    int *d_results, void *d_final_A, void *d_final_B, void *d_final_Z);
/* same with DEVICE buffers in boundary format (inputs resident in HBM, proofs left in HBM) */
int sipp_prove_native_batch_device(const void *dA, const void *dB, size_t n, size_t count, void *d_proofs);
/* sipp_prove_native_batch plus every instance's statement members, as sipp_prove_native_statement gives them for one instance:
 * final_A (count x 64 B), final_B (count x 128 B), final_Z (count x 384 B), byte-identical to sipp_verify_native on
 * (A_j, B_j, proof_j), each may be NULL.  No verification is performed; pairing(final_A, final_B) == final_Z by construction.
 *   - The proofs are those of sipp_prove_native_batch.  Argument checks and codes as for it (a NULL A, B or proofs, count == 0, n
 *     not a non-zero power of two: SIPP_ERR_ARG), all before the device is touched, and valid arguments without a device give
 *     SIPP_ERR_CUDA.  One difference: sipp_prove_native_batch initialises the device first, so without a device it returns
 *     SIPP_ERR_CUDA for bad arguments too, where this call returns SIPP_ERR_ARG.  A bad point or a zero challenge fails the whole
 *     call, and then nothing is written to the proofs or the finals.  Options: those of sipp_prove_native_batch.
 *   - After the last round every instance's first point is its final point; final_Z is one batched one-pair product per instance
 *     (the last step of sipp_verify_native_batch).  sipp_stats: miller_pairs and fold_points grow exactly as for
 *     sipp_prove_native_batch, plus miller_pairs by count when final_Z is non-NULL; launches grows by more (not part of the
 *     contract). */
int sipp_prove_native_batch_statement(const uint8_t *A, const uint8_t *B, size_t n, size_t count, uint8_t *proofs,
                                      uint8_t *final_A, uint8_t *final_B, uint8_t *final_Z);
/* the same with A, B, proofs and the finals in DEVICE memory (boundary format) */
int sipp_prove_native_batch_statement_device(const void *dA, const void *dB, size_t n, size_t count, void *d_proofs,
                                             void *d_final_A, void *d_final_B, void *d_final_Z);

/* ---- batched instances of different sizes: `count` independent proofs in lock-step, each with its own n ------------------- */
/* count independent proofs of instances of different sizes, in lock-step.  Instance j = pairs [offsets[j], offsets[j+1]) of A and B;
 * n_j = offsets[j+1] - offsets[j] must be a non-zero power of two.  offsets: count + 1 HOST entries, offsets[0] = 0, offsets[count] = a_len.
 * proofs: sum_j sipp_proof_len(n_j) x 384 B.  Instance j's proof starts at byte 384 * sum_{k<j} sipp_proof_len(n_k), in the returned
 * (reversed) order.  Every proof is byte-identical to sipp_prove_native on that instance's pairs (prover_native.rs:26-80).
 *   - a_len != b_len: SIPP_ERR_LENGTH.  SIPP_ERR_ARG: a NULL pointer, count == 0, offsets[0] != 0, decreasing offsets,
 *     offsets[count] != a_len, a segment of length 0 or not a power of two, more than 2^32 - 1 pairs.  All of these are returned
 *     before the device is touched; valid arguments without a device give SIPP_ERR_CUDA.
 *   - a coordinate >= p, or with SIPP_OPT_VALIDATE_POINTS a point off the curve or a G2 point outside the subgroup, fails the whole
 *     call with SIPP_ERR_ENCODING, a zero challenge with SIPP_ERR_ZERO_CHALLENGE; in both cases nothing is written to `proofs`.
 *   - n_j = 1 gives the proof [Z] = [pairing(A_i, B_i)].
 *   - Rounds run together: round 0 computes Z of every instance, round r >= 1 the instances with log2 n_j >= r.  The products use
 *     the path of sipp_inner_product_batch.  Options read: SIPP_OPT_FE_NORMALISATION, SIPP_OPT_FQ12_ORDER, SIPP_OPT_WIDE_LINES_MAX,
 *     SIPP_OPT_FE_ENGINE, SIPP_OPT_WIDE_FOLD_MAX, SIPP_OPT_BATCH_KPG_MAX, SIPP_OPT_FOLD_STRAUS, SIPP_OPT_VALIDATE_POINTS and
 *     SIPP_OPT_PRODUCT_CHUNK_PAIRS.  Not read: SIPP_OPT_PIPELINE, SIPP_OPT_BATCH_STREAMS, SIPP_OPT_BATCH_QLINES and the matrix
 *     stages (SIPP_OPT_MATRIX_*).
 *   - The registration of A and B in every instance's transcript is a chain of 8 n_j Poseidon permutations on the device, and the
 *     longest instance bounds it (about 9.4 us per permutation on the device against 0.61 us on the host): an instance far larger
 *     than the rest is better proved on its own with sipp_prove_native.
 *   - sipp_stats.miller_pairs grows by sum_j (3 n_j - 2), fold_points by sum_j (n_j - 1).
 * sipp_verify_native_batch_ragged checks such proofs in one call. */
int sipp_prove_native_batch_ragged(const uint8_t *A, size_t a_len, const uint8_t *B, size_t b_len, const size_t *offsets, size_t count,
                                   uint8_t *proofs);
/* the same with A, B and proofs in DEVICE memory (boundary format); offsets stay on the host */
int sipp_prove_native_batch_ragged_device(const void *dA, const void *dB, size_t n, const size_t *offsets, size_t count, void *d_proofs);
/* sipp_prove_native_batch_ragged plus every instance's statement members, in the caller's instance order: final_A + 64 j,
 * final_B + 128 j, final_Z + 384 j, byte-identical to sipp_verify_native on (A_j, B_j, proof_j), each may be NULL.  No verification
 * is performed; pairing(final_A, final_B) == final_Z by construction.
 *   - The proofs are those of sipp_prove_native_batch_ragged.  Argument checks, their order and codes as for it, all before the
 *     device is touched (valid arguments without a device: SIPP_ERR_CUDA).  A bad point or a zero challenge fails the whole call,
 *     and then nothing is written to the proofs or the finals.  Options: those of sipp_prove_native_batch_ragged.
 *   - After the last round the final points are gathered and paired as sipp_verify_native_batch_ragged does: one batched one-pair
 *     product per instance.  sipp_stats: miller_pairs and fold_points grow exactly as for sipp_prove_native_batch_ragged, plus
 *     miller_pairs by count when final_Z is non-NULL; launches grows by more (not part of the contract). */
int sipp_prove_native_batch_ragged_statement(const uint8_t *A, size_t a_len, const uint8_t *B, size_t b_len, const size_t *offsets,
                                             size_t count, uint8_t *proofs, uint8_t *final_A, uint8_t *final_B, uint8_t *final_Z);
/* the same with A, B, proofs and the finals in DEVICE memory (boundary format); offsets stay on the host */
int sipp_prove_native_batch_ragged_statement_device(const void *dA, const void *dB, size_t n, const size_t *offsets, size_t count,
                                                    void *d_proofs, void *d_final_A, void *d_final_B, void *d_final_Z);
/* count independent verifications of instances of different sizes, in lock-step (verifier_native.rs:14-85 per instance).  A, B,
 * offsets: as for sipp_prove_native_batch_ragged, with the same checks in the same order.  proof_offsets: count + 1 HOST entries in
 * Fq12 units, proof_offsets[0] = 0, never decreasing: proof j is the Fq12 elements [proof_offsets[j], proof_offsets[j+1]) of
 * `proofs` (384 B each), read from its end like the reference's pop() -- its last element is Z, and only its last sipp_proof_len(n_j)
 * elements are read, so a longer proof is accepted as by sipp_verify_native.  The running sums of sipp_proof_len(n_j) give exactly
 * the layout sipp_prove_native_batch_ragged writes.
 *   results[j] = SIPP_OK for Ok(statement), SIPP_ERR_VERIFY for Err("Verification failed"), SIPP_ERR_ENCODING for a coordinate >= p
 *   among the elements read: what sipp_verify_native returns on instance j's pairs and proof slice.  One failed instance does not
 *   affect the others.  For every instance with SIPP_OK or SIPP_ERR_VERIFY, final_A + 64 j, final_B + 128 j and final_Z + 384 j
 *   (when non-NULL) receive its statement members, byte-identical to sipp_verify_native's, in the caller's order.
 *   - The return value reports whether the batch ran, not whether the proofs verified.  a_len != b_len: SIPP_ERR_LENGTH.
 *     SIPP_ERR_ARG: a NULL A, B, offsets, proofs, proof_offsets or results, count == 0, bad offsets (as above), proof_offsets[0] != 0
 *     or decreasing proof_offsets.  A proof shorter than sipp_proof_len(n_j): SIPP_ERR_SHORT_PROOF (verifier_native.rs:31,40,42).
 *     All of these are returned before the device is touched; valid arguments without a device give SIPP_ERR_CUDA.
 *   - a coordinate >= p in A or B, or with SIPP_OPT_VALIDATE_POINTS a point off the curve or a G2 point outside the subgroup, fails
 *     the whole call with SIPP_ERR_ENCODING, a zero challenge with SIPP_ERR_ZERO_CHALLENGE; in both cases nothing is written to
 *     `results` or the finals.
 *   - n_j = 1 gives results[j] = SIPP_OK exactly when pairing(A_i, B_i) == Z.
 *   - The transcripts are replayed first; then the folds of every round run back to back, and every GT update Z_L^x, Z_R^(1/x) of
 *     every instance is one independent power in a single launch beside them.  Options read: SIPP_OPT_FE_NORMALISATION,
 *     SIPP_OPT_FQ12_ORDER, SIPP_OPT_WIDE_LINES_MAX, SIPP_OPT_FE_ENGINE, SIPP_OPT_WIDE_FOLD_MAX, SIPP_OPT_BATCH_KPG_MAX,
 *     SIPP_OPT_FOLD_STRAUS, SIPP_OPT_VALIDATE_POINTS and SIPP_OPT_PRODUCT_CHUNK_PAIRS.  Not read: SIPP_OPT_PIPELINE,
 *     SIPP_OPT_BATCH_STREAMS, SIPP_OPT_BATCH_QLINES and the matrix stages (SIPP_OPT_MATRIX_*).
 *   - As for the prover, the registration of A and B is a device chain of 8 n_j Poseidon permutations per instance, and the longest
 *     instance bounds the call: an instance far larger than the rest is better verified on its own with sipp_verify_native.
 *   - sipp_stats.fold_points grows by sum_j (n_j - 1), miller_pairs by count (the final pairings). */
int sipp_verify_native_batch_ragged(const uint8_t *A, size_t a_len, const uint8_t *B, size_t b_len, const size_t *offsets, size_t count,
                                    const uint8_t *proofs, const size_t *proof_offsets, int *results, uint8_t *final_A, uint8_t *final_B,
                                    uint8_t *final_Z);
/* sipp_verify_native_batch_ragged with A, B, the proofs, d_results (count x int32) and the finals in DEVICE memory (boundary format,
 * 4-byte aligned; n pairs); offsets and proof_offsets stay on the host.  results[j] and every final are byte-identical to the host
 * form's on the same bytes and options: the finals of an instance are written only when its result is SIPP_OK or SIPP_ERR_VERIFY,
 * and its slots are left untouched for SIPP_ERR_ENCODING.  A, B and the proofs are only read, in place.  Argument checks, their order
 * and codes as for the host form, all before the device is touched (valid arguments without a device: SIPP_ERR_CUDA).  A bad point or
 * a zero challenge fails the whole call and writes nothing to d_results or the finals.  Stream order, options and sipp_stats as for
 * sipp_verify_native_batch_device. */
int sipp_verify_native_batch_ragged_device(const void *dA, const void *dB, size_t n, const size_t *offsets, size_t count,
                                           const void *d_proofs, const size_t *proof_offsets, int *d_results, void *d_final_A,
                                           void *d_final_B, void *d_final_Z);

/* ---- input producers of the BLS-aggregation demo (bin/bls_aggregation.rs:95-117; SURVEY 8f row 3) ---------------------------- */
/* Scalars are 32-byte little-endian integers < r.  The `_device` forms take DEVICE pointers in the same formats.
 * `map_to_g2_without_cofactor_mul(u).mul_by_cofactor()` (:100-104) is not provided: it lives in the un-vendored starky-bn254
 * crate and has no specification offline. */
/* public_keys[i] = (G1Affine::generator() * sk_i).into()                  :96-99   -> out: count x 64 B */
int sipp_g1_generator_mul_batch(const uint8_t *scalars, size_t count, uint8_t *out);
int sipp_g1_generator_mul_batch_device(const void *d_scalars, size_t count, void *d_out);
/* signatures[i] = (m_i * sk_i).into()                                     :105-109 -> out: count x 128 B
 * point_count = count: one point per scalar; point_count = 1: every scalar multiplies points[0] (window table, no doublings) */
int sipp_g2_mul_batch(const uint8_t *points, size_t point_count, const uint8_t *scalars, size_t count, uint8_t *out);
int sipp_g2_mul_batch_device(const void *d_points, size_t point_count, const void *d_scalars, size_t count, void *d_out);
/* signatures.iter().fold(G2Projective::zero(), |acc, &s| acc + s).into()  :110-113 -> out: 128 B (count = 0: the identity) */
int sipp_g2_sum(const uint8_t *points, size_t count, uint8_t out[128]);
int sipp_g2_sum_device(const void *d_points, size_t count, void *d_out);
/* -G1Affine::generator()                                                  :116 (host only) */
int sipp_g1_neg_generator(uint8_t out[64]);

/* ---- synthetic inputs and instrumentation --------------------------------------------------------------- */
/* A_i = [a_i]G1, B_i = [b_i]G2 with the documented SplitMix64 scalar stream (same as oracle_seeded_inputs), generated on the
 * GPU by the producers above (keygen over the window tables of the two generators) into DEVICE buffers dA (n x 64 B),
 * dB (n x 128 B) in boundary format */
int sipp_seeded_inputs_device(uint64_t seed, size_t n, void *dA, void *dB);
int sipp_seeded_inputs(uint64_t seed, size_t n, uint8_t *A, uint8_t *B);

typedef struct {
    uint64_t launches;          /* kernels launched since the last reset */
    uint64_t miller_pairs;      /* Miller loops the kernels computed: pairs pushed through the line + accumulation kernels (a pairing-matrix
                                   stage computes more of them than the reference's 3n - 2, see SIPP_OPT_MATRIX_*) */
    uint64_t miller_launches;
    double miller_ms;           /* CUDA-event time of the Miller-loop kernels (SIPP_OPT_PROFILE = 1) */
    double reduce_fe_ms;        /* product reduction + final exponentiation */
    double fold_ms;             /* G1 + G2 fold kernels */
    uint64_t fold_points;       /* folded indices (one G1 + one G2 output each) */
    double transcript_ms;       /* host Poseidon time on the critical path */
    double other_ms;
} sipp_stats;
int sipp_get_stats(sipp_stats *out);
int sipp_reset_stats(void);

/* ---- test / benchmark hooks (exercise single device functions so every layer can be checked against the oracle) -- */
/* op: 0 fq_mul (PTX carry chains), 1 fq_mul (portable), 2 add, 3 sub, 4 inv, 5 neg; elements 32 B */
int sipp_test_fq_op(int op, const uint8_t *a, const uint8_t *b, uint8_t *out, size_t count);
/* op: 0 mul, 1 sqr, 2 inv, 3..5 frobenius^1..3, 6 conj, 7 cyclotomic sqr, 8 cyclotomic ^x; elements 384 B.
 * op + 20 runs the 6-lane cooperative version (29 = cooperative final exponentiation) */
int sipp_test_fq12_op(int op, const uint8_t *a, const uint8_t *b, uint8_t *out, size_t count);
/* host only (no GPU needed): the per-round recoding of the challenge handed to the fold kernel -- GLV (G1, x) and GLS
 * (G2, x^-1) sub-scalars in non-adjacent form.  Writes the raw plan as 32-bit words: 6 components (2 for G1, then 4 for
 * G2) of {plus[5], minus[5], neg}, then g1_bits, g2_bits; returns the number of words written or a negative status. */
int sipp_test_fold_plan(const uint8_t x[32], const uint8_t x_inv[32], uint32_t *out_words, size_t out_cap);
/* the same recoding by the device code of the batched prover's transcript (glv::plan_build with the __device__ tables of
 * k_tr_round), one thread per pair, on `count` pairs (x, x_inv: count x 32 B).  Writes count plans of 68 words in the layout of
 * sipp_test_fold_plan; returns the number of pairs the recoding refused, or a negative status.  The scalars are not checked. */
int sipp_test_fold_plan_device(const uint8_t *x, const uint8_t *x_inv, size_t count, uint32_t *out_words);
/* one launch of a batched fold kernel over `count` instances of n points each (n even): instance j owns A, B [j n, (j + 1) n) and is
 * folded with xs[j], x_invs[j] (32 B each, the checks of sipp_ctx_fold), h = n / 2.  kernel: 0 k_fold_batch, 1 k_fold_wide_batch,
 * 2 k_fold_straus.  Points are decoded and checked as by sipp_ctx_create; A_out (count x h x 64 B), B_out (count x h x 128 B)
 * receive the first h points of every instance. */
int sipp_test_fold_batch(const uint8_t *A, const uint8_t *B, size_t n, size_t count, const uint8_t *xs, const uint8_t *x_invs, int kernel,
                         uint8_t *A_out, uint8_t *B_out);
/* which: 0 mad.lo.u32 chains, 1 mad.wide.u32 chains, 2 lo/hi carry chains, 3 fq_mul PTX, 4 fq_mul portable.
 * returns operations per second (IMAD instructions for 0-2, Fq multiplications for 3-4) in *ops_per_s */
/* device transcript (k_transcript.cu): `count` independent Poseidon permutations, 12 x u64 each, in place */
int sipp_test_poseidon_device(uint64_t *states, size_t count);
/* one transcript round for `count` instances: states in/out (4 x u64 each); fq12s = count x nf x 384 B with nf = 2 (Z_L, Z_R)
 * or 3 (Z, Z_L, Z_R: first round); x_out = count x 64 B (challenge x || x^-1); plans_out = count x raw fold plan
 * (same words as sipp_test_fold_plan) or NULL */
int sipp_test_transcript_round_device(uint64_t *states, const uint8_t *fq12s, int nf, size_t count, uint8_t *x_out, uint32_t *plans_out);
/* host copy of the binary Fr inversion used by the device transcript (glv_core.h): 0 ok, -1 x >= r, -2 x == 0; no GPU needed */
int sipp_test_fr_inverse_binary(const uint8_t x[32], uint8_t out[32]);
int sipp_microbench(int which, int iters, double *ops_per_s, double *ms);
/* host Poseidon self-checks (no GPU): a chain of `count` permutations by the AVX-512 and the portable code side by side, index of the
 * first mismatch or -1; the scalar helpers of the AVX-512 file on crafted operands (which = 0: (in[0] + 2^64 in[1]) mod p; 1: the closing
 * multiply-add of a partial round, in = lo, hi, top, p7, m00; 2: out[0] = in[0]^7, out[1] = in[0]^7 + in[1]; 3, 4: pieces of the IFMA path, see transcript.cc); -1 without AVX-512 / IFMA */
/* the pairing-matrix stage policy (host logic only): blocks of the first stage (which = 0) or of a later stage (which = 1) at n points; 0 = none */
long sipp_test_stage_blocks(int which, size_t n);
/* the plan of sipp_inner_product_batch (host logic only): the accumulator groups of `count` segments (offsets as there) with
 * SIPP_OPT_BATCH_KPG_MAX = kpg_max and SIPP_OPT_PRODUCT_CHUNK_PAIRS = chunk_pairs.  Writes 4 words per group -- first pair, pairs,
 * segment, chunk -- to `out` when out_cap >= 4 x groups, the pairs per group at most to *kpg_out (may be NULL); returns the number
 * of groups or a negative sipp_status */
long sipp_test_product_plan(const size_t *offsets, size_t count, int kpg_max, size_t chunk_pairs, size_t *out, size_t out_cap, int *kpg_out);
/* the schedule of sipp_prove_native_batch_ragged (host logic only) under the current options: 5 words per round r = 0 .. log2 max n_j --
 * active instances, pairs of its products, fold elements, fold kernel (-1 none, 0 k_fold_batch, 1 k_fold_wide_batch, 2 k_fold_straus,
 * in their ragged forms) and line-table chunks -- to `out` when out_cap >= 5 x rounds; returns the number of rounds or a negative
 * sipp_status (the argument checks of sipp_prove_native_batch_ragged) */
long sipp_test_ragged_schedule(const size_t *offsets, size_t count, long long *out, size_t out_cap);
/* the plan of sipp_g1_msm_batch / sipp_g2_msm_batch (host logic only): 4 words per segment -- G1 path (0 Straus, 1 Pippenger), G1 window
 * bits (0 for Straus), G2 path, G2 window bits -- to `out` when out_cap >= 4 x count; returns count or a negative sipp_status (the
 * offsets checks of the entry points) */
long sipp_test_msm_plan(const size_t *offsets, size_t count, int *out, size_t out_cap);
/* sipp_g1_msm_batch_device (group 1) / sipp_g2_msm_batch_device (group 2) with every non-empty segment forced onto one path: c = 0 Straus,
 * 5 <= c <= 16 Pippenger with c-bit windows (another c or group: SIPP_ERR_ARG).  The outputs are the same bytes; for timing both paths
 * at one segment length (tools/msm_time.py). */
int sipp_test_msm_batch_device(int group, int c, const void *d_points, const void *d_scalars, size_t n, const size_t *offsets, size_t count,
                               void *d_out);
/* the plan of sipp_gt_msm_batch (host logic only): 2 words per segment -- path (0 short, 1 Pippenger), window bits (0 for the short
 * path) -- to `out` when out_cap >= 2 x count; returns count or a negative sipp_status (the offsets checks of the entry points) */
long sipp_test_gt_msm_plan(const size_t *offsets, size_t count, int *out, size_t out_cap);
/* sipp_gt_msm_batch_device with every non-empty segment forced onto one path: c = 0 the short path, 2 <= c <= 16 Pippenger with c-bit
 * windows (another c: SIPP_ERR_ARG).  The outputs are the same bytes; for timing both paths at one segment length (tools/gt_msm_time.py). */
int sipp_test_gt_msm_batch_device(int c, const void *d_elems, const void *d_scalars, size_t n, const size_t *offsets, size_t count, void *d_out);
long sipp_test_poseidon_chain(uint64_t seed, long count);
int sipp_test_poseidon_scalar(int which, const uint64_t *in, uint64_t *out);
/* the derived tables of the host Poseidon (sipp::PoseidonFastTables, poseidon_fast.h), for tools/probe/poseidon_lab.cc */
const void *sipp_test_poseidon_tables(void);

#ifdef __cplusplus
}
#endif
#endif

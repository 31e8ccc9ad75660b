// launch.h -- host-callable launch wrappers of the kernels (one translation unit per kernel group so that the
// groups compile in parallel).  Every wrapper returns the cudaError_t of the launch as an int (0 = success).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "fold_plan.h"

namespace sipp {

// Product `y` of a launch pairs A[a_off[y] + j] with B[b_off[y] + j], j < m.
struct MillerJob {
    size_t a_off[2];
    size_t b_off[2];
    size_t m;
};
// Lock-step batch of independent instances: instance `inst` owns points [inst * stride, inst * stride + current n) of A and B;
// product P = inst * nprod + y pairs A[inst * stride + a_off[y] + i] with B[inst * stride + b_off[y] + i], i < h.
struct BatchJob {
    size_t stride;
    size_t a_off[2];
    size_t b_off[2];
    size_t h;
    int nprod;
};
struct Scalar256 {
    uint32_t w[8];
};

#define SIPP_MILLER_BLOCK 64

int launch_codec_decode(const uint32_t* in, uint32_t* out, size_t n_fq, int* flags, cudaStream_t s);
int launch_codec_encode(const uint32_t* in, uint32_t* out, size_t n_fq, cudaStream_t s);
int launch_miller_block(const uint32_t* A, const uint32_t* B, const MillerJob& job, int nprod, uint32_t* partials, cudaStream_t s);
int launch_reduce_fe(const uint32_t* partials, int count, int nprod, uint32_t* out, int final_exp, int ark_norm, cudaStream_t s);
int launch_gt_fold(const uint32_t* in, const Scalar256& x, const Scalar256& xinv, uint32_t* out, cudaStream_t s);
int launch_gt_fold_eng(const uint32_t* in, const Scalar256& x, const Scalar256& xinv, uint32_t* out, cudaStream_t s);
int launch_gt_fold_rounds(const uint32_t* elems, const uint32_t* scalars, int rounds, uint32_t* partials, cudaStream_t s);
int launch_fold(uint32_t* A, uint32_t* B, size_t h, const FoldPlan& plan, cudaStream_t s);
int launch_fold_wide(uint32_t* A, uint32_t* B, size_t h, const FoldPlan& plan, cudaStream_t s);
// on-curve + G2 subgroup check of decoded points: flags |= 2 (off the curve), |= 4 (outside the prime-order subgroup)
int launch_validate_points(const uint32_t* dA, const uint32_t* dB, size_t n, int* flags, cudaStream_t s);
int launch_test_fq_op(int op, const uint32_t* a, const uint32_t* b, uint32_t* out, size_t count, cudaStream_t s);
int launch_test_fq12_op(int op, const uint32_t* a, const uint32_t* b, uint32_t* out, size_t count, cudaStream_t s);
int launch_microbench(int which, int blocks, int threads, void* out, int iters, uint32_t seed, double* ops_per_thread, cudaStream_t s);

// split Miller pipeline (k_coop.cu)
int launch_lines(const uint32_t* A, const uint32_t* B, const MillerJob& job, int nprod, size_t c0, size_t mc, uint32_t* lines, cudaStream_t s);
int launch_lines_wide(const uint32_t* A, const uint32_t* B, const MillerJob& job, int nprod, size_t c0, size_t mc, uint32_t* lines, cudaStream_t s);
int accum_blocks(size_t m_chunk, int kpg);
int launch_accum(const uint32_t* lines, size_t m_chunk, int nprod, int kpg, uint32_t* partials, int block_offset, cudaStream_t s);
int launch_reduce_fe_coop(const uint32_t* partials, int count, int nprod, uint32_t* out, int final_exp, int ark_norm, cudaStream_t s);
int launch_reduce_fe_eng(const uint32_t* partials, int count, int nprod, uint32_t* out, int final_exp, int ark_norm, cudaStream_t s);
int accum_eng_blocks(size_t m_chunk, int kpg);
int launch_accum_eng(const uint32_t* lines, size_t m_chunk, int nprod, int kpg, uint32_t* partials, int block_offset, cudaStream_t s);
int launch_accum_eng_each(const uint32_t* lines, size_t m, uint32_t* out, cudaStream_t s);
int launch_test_coop_op(int op, const uint32_t* a, const uint32_t* b, uint32_t* out, size_t count, cudaStream_t s);
size_t lines_bytes_per_pair();

// pairing-matrix tail (k_mat.cu): E[i][j] = e(A_i, B_j) for the n points left, then folds of the MATRIX instead of the points
int launch_mat_gather(const uint32_t* A, const uint32_t* B, size_t nr, size_t m, uint32_t* Aexp, uint32_t* Bexp, cudaStream_t s);
int launch_mat_fe(const uint32_t* miller, size_t count, uint32_t* E, int ark_norm, cudaStream_t s);
int launch_mat_diag(const uint32_t* E, size_t n, int main_diagonal, uint32_t* partials, cudaStream_t s);
int launch_mat_fold(const uint32_t* E, size_t n, uint32_t* Eout, const GtPlan& plan, cudaStream_t s);

// batched instances (k_coop.cu, k_fold.cu, k_transcript.cu)
int launch_lines_batch(const uint32_t* A, const uint32_t* B, const BatchJob& job, size_t p0, size_t np, uint32_t* lines, cudaStream_t s);
int launch_accum_batch(const uint32_t* lines, size_t pairs, int kpg, uint32_t* partials, size_t group_offset, cudaStream_t s);
int launch_fe_batch(const uint32_t* partials, size_t nproducts, int gpp, int nprod, uint32_t* out, size_t out_stride, int slot0, int slot1, int ark_norm,
                    cudaStream_t s);
int launch_lines_wide_batch(const uint32_t* A, const uint32_t* B, const BatchJob& job, size_t p0, size_t np, uint32_t* lines, cudaStream_t s);
int launch_qlines_batch(const uint32_t* B, size_t npoints, uint32_t* qlines, cudaStream_t s);
int launch_eval_lines_batch(const uint32_t* A, const uint32_t* B, const BatchJob& job, size_t p0, size_t np, const uint32_t* qlines, uint32_t* lines,
                            cudaStream_t s);
size_t qlines_bytes_per_point();
int launch_eval_lines_mat(const uint32_t* A, const uint32_t* B, size_t nr, size_t m, const uint32_t* qlines, uint32_t* lines, cudaStream_t s);
int launch_fe_batch_eng(const uint32_t* partials, size_t nproducts, int gpp, int nprod, uint32_t* out, size_t out_stride, int slot0, int slot1, int ark_norm,
                        cudaStream_t s);
int launch_fold_batch(uint32_t* A, uint32_t* B, size_t h, size_t stride, size_t count, const FoldPlan* plans, cudaStream_t s);
int launch_fold_wide_batch(uint32_t* A, uint32_t* B, size_t h, size_t stride, size_t count, const FoldPlan* plans, cudaStream_t s);
int launch_fold_straus(uint32_t* A, uint32_t* B, size_t h, size_t stride, size_t count, const FoldPlan* plans, cudaStream_t s);
int launch_tr_absorb_pairs(const uint32_t* bytesA, const uint32_t* bytesB, size_t n, size_t count, uint64_t* states, cudaStream_t s);
int launch_tr_round(uint64_t* states, const uint32_t* proofs, size_t np, int slot_z, int slot_l, int slot_r, int order, size_t count, FoldPlan* plans,
                    uint64_t* challenges, int* flags, cudaStream_t s);
int launch_test_poseidon(uint64_t* states, size_t count, cudaStream_t s);
int launch_test_plan_build(const uint64_t* xs, const uint64_t* xinvs, size_t count, FoldPlan* plans, int* fails, cudaStream_t s);
int launch_gt_fold_batch(const uint32_t* proofs, size_t stride, int slot_l, int slot_r, const uint64_t* challenges, uint32_t* z, size_t count,
                         cudaStream_t s);

// batched independent products (k_products.cu, host driver products.cu).  An accumulator group folds pairs [first, first + pairs)
// of the flat pair list, all of one segment and one chunk; a task multiplies work[src .. src + n) into work[dst] (Fq12 slots of 96 words).
struct ProductGroup {
    uint32_t first, pairs;
};
struct ProductTask {
    uint32_t src, n, dst, pad;
};
#define SIPP_PRODUCT_SPAN 40  // Fq12 per task: 2 for each of the 20 six-lane groups of a block
int launch_accum_plan(const uint32_t* lines, const ProductGroup* plan, size_t g0, size_t ngroups, size_t c0, int kpg, uint32_t* partials, cudaStream_t s);
int launch_seg_product(const ProductTask* tasks, size_t ntasks, uint32_t* work, cudaStream_t s);

// ragged batched prover (host driver ragged.cu).  One entry per active instance of a round, in the round's order: its points are
// [base, base + 2h) of the flat arrays, its fold elements [estart, estart + h) of the round, its wide-fold units start at ustart
// (h / 2 units of two elements, or one unit when h = 1).  Round 1's table also gives the absorb: pairs [base, base + 2h).
struct RaggedInst {
    uint32_t estart, ustart, h, base;
};
// proof of an instance: Fq12 slots [first, first + np) of the flat proof buffer
struct RaggedProof {
    uint64_t first;
    uint32_t np, pad;
};
int launch_fold_batch_ragged(uint32_t* A, uint32_t* B, const RaggedInst* tab, unsigned act, size_t elems, const FoldPlan* plans, cudaStream_t s);
int launch_fold_wide_batch_ragged(uint32_t* A, uint32_t* B, const RaggedInst* tab, unsigned act, size_t elems, size_t units, const FoldPlan* plans,
                                  cudaStream_t s);
int launch_fold_straus_ragged(uint32_t* A, uint32_t* B, const RaggedInst* tab, unsigned act, size_t elems, const FoldPlan* plans, cudaStream_t s);
int launch_tr_absorb_pairs_ragged(const uint32_t* bytesA, const uint32_t* bytesB, const RaggedInst* tab, unsigned act, uint64_t* states, cudaStream_t s);
// challenges: NULL, or act x 8 u64 (x || x^-1 of every active instance)
int launch_tr_round_ragged(uint64_t* states, const uint32_t* proofs, const RaggedProof* pt, int round, int order, unsigned act, FoldPlan* plans,
                           uint64_t* challenges, int* flags, cudaStream_t s);
// gA / gB <- per active instance A_hi || A_lo and B_lo || B_hi at pairs [2 estart, 2 estart + 2h): Z_L and Z_R as two segments
int launch_ragged_gather(const uint32_t* A, const uint32_t* B, const RaggedInst* tab, unsigned act, size_t elems, uint32_t* gA, uint32_t* gB, cudaStream_t s);
// proofs[dst[j]] <- res[j] (Fq12 slots of 96 words)
int launch_scatter_fq12(const uint32_t* res, const uint64_t* dst, size_t count, uint32_t* proofs, cudaStream_t s);

// ragged batched verifier (host driver ragged.cu).  A GT entry: a power entry e reads Z_L at Fq12 slot `src` of the proofs and Z_R at
// src - 1, with challenges[8 e .. 8 e + 8) = x || x^-1, and writes Z_L^x Z_R^(1/x) to factor slot `dst`; a Z entry copies the Fq12 at
// `src` (decoded) to factor slot `dst`.  Factor slots are Fq12 of 96 words in the layout of k_seg_product.
struct RaggedGt {
    uint64_t src;
    uint32_t dst, pad;
};
// entries [0, npow) are powers, [npow, npow + nz) Z copies
int launch_gt_fold_ragged(const uint32_t* proofs, const RaggedGt* ent, size_t npow, size_t nz, const uint64_t* challenges, uint32_t* factors, cudaStream_t s);
// gA[j] <- A[at[j]], gB[j] <- B[at[j]] (decoded points), j < count
int launch_gather_points(const uint32_t* A, const uint32_t* B, const uint64_t* at, size_t count, uint32_t* gA, uint32_t* gB, cudaStream_t s);

// BLS input producers (k_bls.cu): group 1 = G1 (16 words per point), 2 = G2 (32 words)
size_t window_table_bytes(int group);
int launch_window_table(int group, const uint32_t* base, uint32_t* table, cudaStream_t s);
int launch_fixed_base_mul(int group, const uint32_t* table, const uint32_t* scalars, size_t count, uint32_t* out, cudaStream_t s);
int launch_g2_mul_var(const uint32_t* points, const uint32_t* scalars, size_t count, uint32_t* out, cudaStream_t s);
int g2_sum_blocks(size_t count, int sm_count);
int launch_g2_sum(const uint32_t* points, size_t count, uint32_t* partials, int blocks, uint32_t* out, cudaStream_t s);
int launch_seeded_scalars(uint64_t seed, size_t n, uint32_t* sa, uint32_t* sb, cudaStream_t s);
int launch_generators(uint32_t* gens, cudaStream_t s);

}  // namespace sipp

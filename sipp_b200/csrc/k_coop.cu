// k_coop.cu -- the split Miller-loop pipeline and the lane-cooperative reduction / final exponentiation.
//
//   k_lines        L: one thread per pair walks the G2 point through the optimal-ate schedule (64 tangents, 25 chords,
//                  2 Frobenius chords) and writes the 91 line functions, already evaluated at P, to HBM:
//                  lines[pair][step] = {l0 yP, l1 xP, xi l1 xP, l3, xi l3}  (5 Fq2 = 320 B; 29,120 B per pair).
//                  Small per-thread state (T, P, Q) -> no spills, Fq2 arithmetic fully inlined.
//   k_accum        A: a group of 6 lanes holds one Fq12 accumulator f in the w-basis (lane k = coefficient of w^k)
//                  and folds the lines of `kpg` pairs into it:  per step  f <- f^2 (once, shared by all kpg pairs)
//                  then f <- f * line for each pair.  Each sparse product is 2 lazy inner products of 6 terms per
//                  lane (fqdot.cuh).  Lines are staged global -> shared with cp.async one line ahead.
//                  Block-level tree product -> one 384 B partial per block.
//   k_reduce_fe_coop  product of the partials and ONE cooperative final exponentiation per product.
//
// Replaces the per-pair `pairing` calls + serial product of /root/reference/src/prover_native.rs:17-22 (and :48-49).
#define SIPP_CURVE_FQ2_CALLS 1
#include "accum.cuh"
#include "coop.cuh"
#include "device_common.cuh"

namespace sipp {

// ------------------------------------------------------------------------------------------------ L: line generation
// A chunk covers pairs [c0, c0 + mc) of EVERY product of the job; lines layout [prod][mc][91][80 words].
__device__ __forceinline__ void lines_of_pair(const G1A& p, const G2A& q, uint32_t* __restrict__ out) {
    if (affine_is_identity(p) || affine_is_identity(q)) {
        // contributes the factor 1: every line is the constant 1
        Fq2 one = fq2_one(), zero = fq2_zero();
        for (int s = 0; s < SIPP_LINES_PER_PAIR; s++) {
            uint32_t* o = out + s * SIPP_LINE_WORDS;
            stream_fq2_words(o, one);
            stream_fq2_words(o + 16, zero);
            stream_fq2_words(o + 32, zero);
            stream_fq2_words(o + 48, zero);
            stream_fq2_words(o + 64, zero);
        }
        return;
    }
    miller_lines(
        p, q, [](int) {},
        [&](int s, const Fq2& l0, const Fq2& l1, const Fq2& l3) {
            uint32_t* o = out + s * SIPP_LINE_WORDS;
            stream_fq2_words(o, l0);
            stream_fq2_words(o + 16, l1);
            stream_fq2_words(o + 32, fq2_mul_xi(l1));
            stream_fq2_words(o + 48, l3);
            stream_fq2_words(o + 64, fq2_mul_xi(l3));
        });
}
#ifndef SIPP_LINES_MINBLOCKS
#define SIPP_LINES_MINBLOCKS 4  // 230 registers; capping at 128 (8 blocks) spills and measured 8% slower (profiles/r01_ab_occupancy.txt)
#endif
__global__ void __launch_bounds__(64, SIPP_LINES_MINBLOCKS) k_lines(const uint32_t* __restrict__ A, const uint32_t* __restrict__ B, MillerJob job, int nprod, size_t c0,
                                              size_t mc, uint32_t* __restrict__ lines) {
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= mc * (size_t)nprod) return;
    int prod = (int)(t / mc);
    size_t j = c0 + (t - (size_t)prod * mc);
    lines_of_pair(load_g1(A, job.a_off[prod] + j), load_g2(B, job.b_off[prod] + j), lines + t * SIPP_PAIR_LINE_WORDS);
}

// Batched instances (lock-step rounds over `count` independent SIPP instances, launch.h BatchJob): product P = inst * nprod + y
// pairs A[inst * stride + a_off[y] + i] with B[inst * stride + b_off[y] + i], i < h.  A chunk covers whole products
// [p0, p0 + np); lines layout [product][h][91][80 words], so one accumulator group owns consecutive pairs of ONE product.
__global__ void __launch_bounds__(64, SIPP_LINES_MINBLOCKS) k_lines_batch(const uint32_t* __restrict__ A, const uint32_t* __restrict__ B, BatchJob job, size_t p0,
                                                                         size_t np, uint32_t* __restrict__ lines) {
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= np * job.h) return;
    size_t P = p0 + t / job.h, i = t % job.h;
    size_t inst = P / (size_t)job.nprod;
    int y = (int)(P % (size_t)job.nprod);
    size_t base = inst * job.stride + i;
    lines_of_pair(load_g1(A, base + job.a_off[y]), load_g2(B, base + job.b_off[y]), lines + t * SIPP_PAIR_LINE_WORDS);
}

// Line coefficients that depend on Q alone.  A line of the Miller loop is (l0 yP, l1 xP, l3) with (l0, l1, l3) functions of the
// G2 point only, and the prover pairs every B_i twice before the first fold: with A_i in Z (prover_native.rs:29) and with its
// cross partner in the first Z_L / Z_R (:48-49).  k_qlines_batch walks each G2 point through the schedule ONCE and keeps
// (l0, l1, l3) (91 x 3 Fq2 = 17,472 B per point); k_eval_lines_batch turns them into the line table of a launch (two Fq2-by-Fq
// scalings per line: 364 of the 3,155 Fq-mul of a full line computation; memory-bound).
#define SIPP_QLINE_WORDS 48
__global__ void __launch_bounds__(64, SIPP_LINES_MINBLOCKS) k_qlines_batch(const uint32_t* __restrict__ B, size_t npoints, uint32_t* __restrict__ qlines) {
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= npoints) return;
    const G2A q = load_g2(B, t);
    if (affine_is_identity(q)) return;  // never read: k_eval_lines_batch writes the constant-1 lines for such a pair
    G1A unit;
    unit.x = fq_one(); unit.y = fq_one();
    uint32_t* out = qlines + t * (size_t)(SIPP_LINES_PER_PAIR * SIPP_QLINE_WORDS);
    miller_lines(
        unit, q, [](int) {},
        [&](int s, const Fq2& l0, const Fq2& l1, const Fq2& l3) {
            uint32_t* o = out + s * SIPP_QLINE_WORDS;
            store_fq2_words(o, l0);
            store_fq2_words(o + 16, l1);
            store_fq2_words(o + 32, l3);
        });
}
// one thread per (pair, step); same pair indexing as k_lines_batch, same output layout as k_lines
__global__ void __launch_bounds__(128) k_eval_lines_batch(const uint32_t* __restrict__ A, const uint32_t* __restrict__ B, BatchJob job, size_t p0, size_t np,
                                                          const uint32_t* __restrict__ qlines, uint32_t* __restrict__ lines) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= np * job.h * SIPP_LINES_PER_PAIR) return;
    const size_t pair = t / SIPP_LINES_PER_PAIR;
    const int step = (int)(t - pair * SIPP_LINES_PER_PAIR);
    const size_t P = p0 + pair / job.h, i = pair % job.h;
    const size_t inst = P / (size_t)job.nprod;
    const int y = (int)(P % (size_t)job.nprod);
    const size_t ia = inst * job.stride + i + job.a_off[y], ib = inst * job.stride + i + job.b_off[y];
    const G1A p = load_g1(A, ia);
    uint32_t* o = lines + t * SIPP_LINE_WORDS;
    // identity test of Q on its first 64 bytes is not enough (x = 0 alone is a valid coordinate): read both halves
    const G2A q = load_g2(B, ib);
    if (affine_is_identity(p) || affine_is_identity(q)) {
        stream_fq2_words(o, fq2_one());
        stream_fq2_words(o + 16, fq2_zero());
        stream_fq2_words(o + 32, fq2_zero());
        stream_fq2_words(o + 48, fq2_zero());
        stream_fq2_words(o + 64, fq2_zero());
        return;
    }
    const uint32_t* src = qlines + (ib * SIPP_LINES_PER_PAIR + step) * SIPP_QLINE_WORDS;
    const Fq2 l0 = fq2_scale(load_fq2_words(src), p.y), l1 = fq2_scale(load_fq2_words(src + 16), p.x), l3 = load_fq2_words(src + 32);
    stream_fq2_words(o, l0);
    stream_fq2_words(o + 16, l1);
    stream_fq2_words(o + 32, fq2_mul_xi(l1));
    stream_fq2_words(o + 48, l3);
    stream_fq2_words(o + 64, fq2_mul_xi(l3));
}

// pairing-matrix stages (k_mat.cu) with many pairs per entry: entry (i, j) of an nr x nr matrix pairs A[i m + t] with B[j m + t],
// t < m, so every B point meets nr different A points -- its line coefficients are computed once (k_qlines_batch) and evaluated
// here.  Pair index q = (i nr + j) m + t, one thread per (pair, step), output layout as k_lines.
__global__ void __launch_bounds__(128) k_eval_lines_mat(const uint32_t* __restrict__ A, const uint32_t* __restrict__ B, size_t nr, size_t m,
                                                        const uint32_t* __restrict__ qlines, uint32_t* __restrict__ lines) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nr * nr * m * SIPP_LINES_PER_PAIR) return;
    const size_t pair = t / SIPP_LINES_PER_PAIR;
    const int step = (int)(t - pair * SIPP_LINES_PER_PAIR);
    const size_t e = pair / m, u = pair % m;
    const size_t ia = (e / nr) * m + u, ib = (e % nr) * m + u;
    const G1A p = load_g1(A, ia);
    uint32_t* o = lines + t * SIPP_LINE_WORDS;
    const G2A q = load_g2(B, ib);
    if (affine_is_identity(p) || affine_is_identity(q)) {
        stream_fq2_words(o, fq2_one());
        stream_fq2_words(o + 16, fq2_zero());
        stream_fq2_words(o + 32, fq2_zero());
        stream_fq2_words(o + 48, fq2_zero());
        stream_fq2_words(o + 64, fq2_zero());
        return;
    }
    const uint32_t* src = qlines + (ib * SIPP_LINES_PER_PAIR + step) * SIPP_QLINE_WORDS;
    const Fq2 l0 = fq2_scale(load_fq2_words(src), p.y), l1 = fq2_scale(load_fq2_words(src + 16), p.x), l3 = load_fq2_words(src + 32);
    stream_fq2_words(o, l0);
    stream_fq2_words(o + 16, l1);
    stream_fq2_words(o + 32, fq2_mul_xi(l1));
    stream_fq2_words(o + 48, l3);
    stream_fq2_words(o + 64, fq2_mul_xi(l3));
}

// ------------------------------------------------------------------------------------------------ A: accumulation
// grid = (blocks, nprod).  Group gid of product `prod` folds pairs [gid * kpg, (gid + 1) * kpg) of that product.
// lines: chunk-local, pair index = prod_local_base + j.
__global__ void __launch_bounds__(SIPP_ACCUM_THREADS, SIPP_ACCUM_MINBLOCKS) k_accum(const uint32_t* __restrict__ lines, size_t m_chunk, int nprod_in_chunk, int kpg,
                                                            uint32_t* __restrict__ partials, int partial_stride_prod, int block_offset, int segmented) {
    __shared__ __align__(16) uint32_t stage[SIPP_ACCUM_GROUPS][2][SIPP_LINE_WORDS];
    __shared__ __align__(16) uint32_t red[SIPP_ACCUM_GROUPS * 96];
    const Lane6 L = lane6_of_thread();
    const int warp = threadIdx.x >> 5;
    const int group = warp * SIPP_GROUPS_PER_WARP + L.base / 6;  // 0..19; idle lanes (30,31) get group index +5: clamp below
    const bool active_lane = L.k < 6;
    const int grp = active_lane ? group : warp * SIPP_GROUPS_PER_WARP;  // idle lanes shadow group 0 of the warp (results unused)
    const int k = active_lane ? L.k : 0;
    const int prod = blockIdx.y;
    const size_t gid = (size_t)blockIdx.x * SIPP_ACCUM_GROUPS + grp;
    const size_t j0 = gid * (size_t)kpg;
    size_t j1 = j0 + (size_t)kpg;
    if (j1 > m_chunk) j1 = m_chunk;
    const int npairs = j0 < m_chunk ? (int)(j1 - j0) : 0;
    const uint32_t* base = lines + ((size_t)prod * m_chunk + j0) * SIPP_PAIR_LINE_WORDS;

    // total line fetches of this group: 91 * npairs, order = step-major (step s, pair q)
    const int total = SIPP_LINES_PER_PAIR * npairs;
    auto line_ptr = [&](int idx) { int s = idx / (npairs > 0 ? npairs : 1); int q = idx - s * (npairs > 0 ? npairs : 1);
                                   return base + (size_t)q * SIPP_PAIR_LINE_WORDS + s * SIPP_LINE_WORDS; };
    auto prefetch = [&](int idx, int buf) {
        if (active_lane && idx < total) {
            const uint32_t* src = line_ptr(idx);
            // 320 B = 20 x 16 B; 6 lanes copy 4 chunks each (24 >= 20)
            for (int c = k; c < 20; c += 6) cp_async16(&stage[grp][buf][c * 4], src + c * 4);
        }
        cp_async_commit();
    };

    Fq2 f = lane_one(k);
    int fetch = 0;
    prefetch(0, 0);
    const unsigned long long plus = SIPP_ATE_PLUS_MASK, minus = SIPP_ATE_MINUS_MASK;
    // every warp runs the full schedule (uniform control flow: shuffles inside); groups without pairs multiply by stale
    // data that is discarded -- their f is reset to 1 at the end
    int maxpairs = kpg;
    auto fold_lines = [&]() {
        for (int q = 0; q < maxpairs; q++) {
            cp_async_wait_all();
            __syncwarp();
            int buf = fetch & 1;
            prefetch(fetch + 1, buf ^ 1);
            Fq2 nf = coop_sparse(L, f, &stage[grp][buf][0]);
            if (q < npairs) { f = nf; fetch++; }
            __syncwarp();
        }
    };
    for (int i = 63; i >= 0; i--) {
        if (i != 63) f = coop_sqr(L, f);
        fold_lines();
        if (((plus | minus) >> i) & 1ull) fold_lines();
    }
    fold_lines();
    fold_lines();
    if (npairs == 0) f = lane_one(k);

    if (segmented) {
        // batched instances: a group's pairs all belong to one product; the per-product reduction (k_fe_batch) multiplies the
        // h / kpg consecutive group results.  block_offset counts groups here.
        if (active_lane && npairs > 0) store_fq2_words(partials + ((size_t)block_offset + gid) * 96 + k * 16, f);
        return;
    }
    f = block_product_coop(L, f, red, active_lane ? group : SIPP_ACCUM_GROUPS, SIPP_ACCUM_GROUPS);
    if (active_lane && group == 0) store_fq2_words(partials + ((size_t)(blockIdx.x + block_offset) * partial_stride_prod + prod) * 96 + k * 16, f);
}

// ------------------------------------------------------------------------------------------------ reduction + final exponentiation
// grid = nprod blocks of 128 threads (20 groups).  partials layout [count][nprod][96].  final_exp = 0 writes the raw
// product in device format (multi-GPU partial), else boundary bytes.
__global__ void __launch_bounds__(SIPP_ACCUM_THREADS) k_reduce_fe_coop(const uint32_t* __restrict__ partials, int count, int nprod,
                                                                     uint32_t* __restrict__ out, int final_exp, int ark_norm) {
    __shared__ __align__(16) uint32_t red[SIPP_ACCUM_GROUPS * 96];
    const Lane6 L = lane6_of_thread();
    const int warp = threadIdx.x >> 5;
    const bool active_lane = L.k < 6;
    const int group = active_lane ? warp * SIPP_GROUPS_PER_WARP + L.base / 6 : SIPP_ACCUM_GROUPS;
    const int k = active_lane ? L.k : 0;
    const int prod = blockIdx.x;
    Fq2 f = lane_one(k);
    int rounds = (count + SIPP_ACCUM_GROUPS - 1) / SIPP_ACCUM_GROUPS;
    for (int r = 0; r < rounds; r++) {
        int i = r * SIPP_ACCUM_GROUPS + group;
        bool have = active_lane && i < count;
        Fq2 v = have ? load_fq2_words(partials + ((size_t)i * nprod + prod) * 96 + k * 16) : lane_one(k);
        f = (r == 0) ? v : coop_mul(L, f, v);
    }
    int live = count < SIPP_ACCUM_GROUPS ? count : SIPP_ACCUM_GROUPS;
    if (live > 1) f = block_product_coop(L, f, red, group, SIPP_ACCUM_GROUPS);
    if (warp == 0) {
        if (final_exp) f = coop_final_exp(L, f, ark_norm != 0);
        if (active_lane && group == 0) {
            if (final_exp) {
                int slot = (k & 1) * 3 + (k >> 1);
                fq2_encode(out + prod * 96 + slot * 16, f);
            } else {
                store_fq2_words(out + prod * 96 + k * 16, f);
            }
        }
    }
}


// Batched instances: product P multiplies its `gpp` consecutive group results and takes ONE final exponentiation; 20 products
// per block (6 lanes each).  out: instance `P / nprod` at out + inst * out_stride words, Fq12 slot slot0 (y = 0) / slot1 (y = 1),
// boundary bytes -- the instance's proof vector, written in its final (reversed) order (prover_native.rs:78).
__global__ void __launch_bounds__(SIPP_ACCUM_THREADS, 3) k_fe_batch(const uint32_t* __restrict__ partials, size_t nproducts, int gpp, int nprod,
                                                               uint32_t* __restrict__ out, size_t out_stride, int slot0, int slot1, int ark_norm) {
    const Lane6 L = lane6_of_thread();
    const int warp = threadIdx.x >> 5;
    const bool active_lane = L.k < 6;
    const int group = warp * SIPP_GROUPS_PER_WARP + (active_lane ? L.base / 6 : 0);
    const int k = active_lane ? L.k : 0;
    size_t P = (size_t)blockIdx.x * SIPP_ACCUM_GROUPS + group;
    const bool have = active_lane && P < nproducts;
    if (P >= nproducts) P = nproducts - 1;
    const uint32_t* src = partials + P * (size_t)gpp * 96 + k * 16;
    Fq2 f = load_fq2_words(src);
    for (int g = 1; g < gpp; g++) f = coop_mul(L, f, load_fq2_words(src + (size_t)g * 96));
    f = coop_final_exp(L, f, ark_norm != 0);
    if (have) {
        size_t inst = P / (size_t)nprod;
        int y = (int)(P % (size_t)nprod);
        int slot = (k & 1) * 3 + (k >> 1);
        fq2_encode(out + inst * out_stride + (size_t)(y ? slot1 : slot0) * 96 + slot * 16, f);
    }
}

// acc <- acc^(2^254) base^e on a 6-lane group (acc = 1: base^e): generic square-and-multiply over the 254 bits of e (4 u64,
// little-endian) -- proof elements need not lie in the cyclotomic subgroup, and the reference's `pow` does not assume it -- with
// the multiplication computed at every bit and selected (groups of one warp hold different exponents).  The accumulator is the
// caller's: returning it by value costs k_gt_fold_batch 64 bytes of stack frame.
__device__ __forceinline__ void coop_pow254(const Lane6& L, const Fq2& base, const uint64_t* e, Fq2& acc) {
#pragma unroll 1
    for (int i = 253; i >= 0; i--) {
        acc = coop_sqr(L, acc);
        const Fq2 m = coop_mul(L, acc, base);
        acc = select_fq2(((e[i >> 6] >> (i & 63)) & 1ull) != 0, m, acc);
    }
}

// Batched verifier GT update (verifier_native.rs:59-61): Z <- Z_L^x * Z * Z_R^(x^-1) for every instance, 6 lanes per power
// (two groups per instance, both in the same block; coop_pow254).  proofs: [count][stride][96] boundary bytes; challenges:
// [count][8] u64 = x || x^-1; z: [count][96] boundary bytes, updated in place.
__global__ void __launch_bounds__(SIPP_ACCUM_THREADS) k_gt_fold_batch(const uint32_t* __restrict__ proofs, size_t stride, int slot_l, int slot_r,
                                                                    const uint64_t* __restrict__ challenges, uint32_t* __restrict__ z, size_t count) {
    __shared__ __align__(16) uint32_t xch[SIPP_ACCUM_GROUPS * 96];
    const Lane6 L = lane6_of_thread();
    const int warp = threadIdx.x >> 5;
    const bool active_lane = L.k < 6;
    const int group = warp * SIPP_GROUPS_PER_WARP + (active_lane ? L.base / 6 : 0);
    const int k = active_lane ? L.k : 0;
    size_t g = (size_t)blockIdx.x * SIPP_ACCUM_GROUPS + group;
    const bool have = active_lane && g < 2 * count;
    if (g >= 2 * count) g = 2 * count - 1;
    const size_t inst = g >> 1;
    const int which = (int)(g & 1);
    const int slot = (k & 1) * 3 + (k >> 1);
    const Fq2 base = fq2_decode(proofs + (inst * stride + (size_t)(which ? slot_r : slot_l)) * 96 + 16 * slot);
    Fq2 acc = lane_one(k);
    coop_pow254(L, base, challenges + 8 * inst + 4 * which, acc);
    if (have && which == 1) store_fq2_words(xch + group * 96 + k * 16, acc);
    __syncthreads();
    // group of Z_L (even g; its partner g + 1 is the next group of the same block: 20 groups per block)
    const Fq2 zr_pow = load_fq2_words(xch + (which == 0 && group + 1 < SIPP_ACCUM_GROUPS ? group + 1 : group) * 96 + k * 16);
    const Fq2 zc = fq2_decode(z + inst * 96 + 16 * slot);
    const Fq2 r = coop_mul(L, coop_mul(L, acc, zc), zr_pow);
    if (have && which == 0) fq2_encode(z + inst * 96 + 16 * slot, r);
}

// Ragged batched verifier (ragged.cu): the GT updates of every round of every instance in ONE launch.  The verifier's challenges
// depend only on A, B and the proof (verifier_native.rs:33-45), so once the transcript has been replayed every Z_L^x, Z_R^(1/x)
// is an independent power and final_Z = Z * prod_r Z_L(r)^x_r Z_R(r)^(1/x_r) (:59-61 unrolled; exact in GT).  Power entry e
// (launch.h RaggedGt): two groups in the same block as in k_gt_fold_batch, Z_L at proofs slot src and Z_R at src - 1, exponents
// challenges[8 e ..] = x || x^-1; their product goes to factors[dst] un-encoded.  The blocks after the powers copy Z of every
// instance (entries npow ..), decoded, to its factor slot, one thread per Fq2 coefficient.  A segmented product finishes.
__global__ void __launch_bounds__(SIPP_ACCUM_THREADS) k_gt_fold_ragged(const uint32_t* __restrict__ proofs, const RaggedGt* __restrict__ ent, size_t npow,
                                                                     size_t nz, const uint64_t* __restrict__ challenges, uint32_t* __restrict__ factors) {
    __shared__ __align__(16) uint32_t xch[SIPP_ACCUM_GROUPS * 96];
    const size_t pow_blocks = (2 * npow + SIPP_ACCUM_GROUPS - 1) / SIPP_ACCUM_GROUPS;
    if (blockIdx.x >= pow_blocks) {  // block-uniform
        const size_t t = (size_t)(blockIdx.x - pow_blocks) * blockDim.x + threadIdx.x;
        if (t >= 6 * nz) return;
        const RaggedGt z = ent[npow + t / 6];
        const int k = (int)(t % 6), slot = (k & 1) * 3 + (k >> 1);
        store_fq2_words(factors + (size_t)z.dst * 96 + k * 16, fq2_decode(proofs + z.src * 96 + 16 * slot));
        return;
    }
    const Lane6 L = lane6_of_thread();
    const int warp = threadIdx.x >> 5;
    const bool active_lane = L.k < 6;
    const int group = warp * SIPP_GROUPS_PER_WARP + (active_lane ? L.base / 6 : 0);
    const int k = active_lane ? L.k : 0;
    size_t g = (size_t)blockIdx.x * SIPP_ACCUM_GROUPS + group;
    const bool have = active_lane && g < 2 * npow;
    if (g >= 2 * npow) g = 2 * npow - 1;
    const size_t e = g >> 1;
    const int which = (int)(g & 1);
    const int slot = (k & 1) * 3 + (k >> 1);
    const RaggedGt en = ent[e];
    const Fq2 base = fq2_decode(proofs + (en.src - (uint64_t)which) * 96 + 16 * slot);
    Fq2 acc = lane_one(k);
    coop_pow254(L, base, challenges + 8 * e + 4 * which, acc);
    if (have && which == 1) store_fq2_words(xch + group * 96 + k * 16, acc);
    __syncthreads();
    const Fq2 zr_pow = load_fq2_words(xch + (which == 0 && group + 1 < SIPP_ACCUM_GROUPS ? group + 1 : group) * 96 + k * 16);
    const Fq2 r = coop_mul(L, acc, zr_pow);
    if (have && which == 0) store_fq2_words(factors + (size_t)en.dst * 96 + k * 16, r);
}

// ------------------------------------------------------------------------------------------------ test hook
// op: 0 mul, 1 sqr (via mul), 2 inv, 3..5 frobenius, 6 conj, 7 cyclotomic sqr, 8 cyclotomic ^x, 9 final exponentiation
__global__ void __launch_bounds__(32) k_test_coop_op(int op, const uint32_t* __restrict__ a, const uint32_t* __restrict__ b, uint32_t* __restrict__ out,
                                                     size_t count) {
    const Lane6 L = lane6_of_thread();
    const bool active_lane = L.k < 6;
    const int k = active_lane ? L.k : 0;
    size_t i = (size_t)blockIdx.x * SIPP_GROUPS_PER_WARP + (active_lane ? L.base / 6 : 0);
    bool have = i < count;
    if (!have) i = count - 1;
    int slot = (k & 1) * 3 + (k >> 1);
    Fq2 x = fq2_decode(a + 96 * i + 16 * slot);
    Fq2 y = b ? fq2_decode(b + 96 * i + 16 * slot) : lane_one(k);
    Fq2 r;
    switch (op) {
        case 0: r = coop_mul(L, x, y); break;
        case 1: r = coop_sqr(L, x); break;
        case 2: r = coop_inv(L, x); break;
        case 3: r = coop_frob(L, x, 1); break;
        case 4: r = coop_frob(L, x, 2); break;
        case 5: r = coop_frob(L, x, 3); break;
        case 6: r = coop_conj(L, x); break;
        case 7: r = coop_cyc_sqr(L, x); break;
        case 8: r = coop_cyc_exp_x(L, x); break;
        default: r = coop_final_exp(L, x, false); break;
    }
    if (have && active_lane) fq2_encode(out + 96 * i + 16 * slot, r);
}

// ------------------------------------------------------------------------------------------------ launch wrappers
int launch_lines(const uint32_t* A, const uint32_t* B, const MillerJob& job, int nprod, size_t c0, size_t mc, uint32_t* lines, cudaStream_t s) {
    size_t threads = mc * (size_t)nprod;
    k_lines<<<(unsigned)((threads + 63) / 64), 64, 0, s>>>(A, B, job, nprod, c0, mc, lines);
    return (int)cudaGetLastError();
}
int accum_blocks(size_t m_chunk, int kpg) {
    size_t groups = (m_chunk + (size_t)kpg - 1) / (size_t)kpg;
    return (int)((groups + SIPP_ACCUM_GROUPS - 1) / SIPP_ACCUM_GROUPS);
}
int launch_accum(const uint32_t* lines, size_t m_chunk, int nprod, int kpg, uint32_t* partials, int block_offset, cudaStream_t s) {
    dim3 grid((unsigned)accum_blocks(m_chunk, kpg), (unsigned)nprod);
    k_accum<<<grid, SIPP_ACCUM_THREADS, 0, s>>>(lines, m_chunk, nprod, kpg, partials, nprod, block_offset, 0);
    return (int)cudaGetLastError();
}
int launch_reduce_fe_coop(const uint32_t* partials, int count, int nprod, uint32_t* out, int final_exp, int ark_norm, cudaStream_t s) {
    k_reduce_fe_coop<<<nprod, SIPP_ACCUM_THREADS, 0, s>>>(partials, count, nprod, out, final_exp, ark_norm);
    return (int)cudaGetLastError();
}
int launch_test_coop_op(int op, const uint32_t* a, const uint32_t* b, uint32_t* out, size_t count, cudaStream_t s) {
    k_test_coop_op<<<(unsigned)((count + SIPP_GROUPS_PER_WARP - 1) / SIPP_GROUPS_PER_WARP), 32, 0, s>>>(op, a, b, out, count);
    return (int)cudaGetLastError();
}
int launch_lines_batch(const uint32_t* A, const uint32_t* B, const BatchJob& job, size_t p0, size_t np, uint32_t* lines, cudaStream_t s) {
    size_t threads = np * job.h;
    k_lines_batch<<<(unsigned)((threads + 63) / 64), 64, 0, s>>>(A, B, job, p0, np, lines);
    return (int)cudaGetLastError();
}
// segmented accumulation of a chunk of `pairs` = products * h pairs, kpg | h; group results to partials[group_offset + gid]
int launch_accum_batch(const uint32_t* lines, size_t pairs, int kpg, uint32_t* partials, size_t group_offset, cudaStream_t s) {
    dim3 grid((unsigned)accum_blocks(pairs, kpg), 1);
    k_accum<<<grid, SIPP_ACCUM_THREADS, 0, s>>>(lines, pairs, 1, kpg, partials, 1, (int)group_offset, 1);
    return (int)cudaGetLastError();
}
int launch_fe_batch(const uint32_t* partials, size_t nproducts, int gpp, int nprod, uint32_t* out, size_t out_stride, int slot0, int slot1, int ark_norm,
                    cudaStream_t s) {
    k_fe_batch<<<(unsigned)((nproducts + SIPP_ACCUM_GROUPS - 1) / SIPP_ACCUM_GROUPS), SIPP_ACCUM_THREADS, 0, s>>>(partials, nproducts, gpp, nprod, out, out_stride,
                                                                                                                slot0, slot1, ark_norm);
    return (int)cudaGetLastError();
}
int launch_gt_fold_batch(const uint32_t* proofs, size_t stride, int slot_l, int slot_r, const uint64_t* challenges, uint32_t* z, size_t count,
                         cudaStream_t s) {
    size_t groups = 2 * count;
    k_gt_fold_batch<<<(unsigned)((groups + SIPP_ACCUM_GROUPS - 1) / SIPP_ACCUM_GROUPS), SIPP_ACCUM_THREADS, 0, s>>>(proofs, stride, slot_l, slot_r, challenges,
                                                                                                                   z, count);
    return (int)cudaGetLastError();
}
int launch_gt_fold_ragged(const uint32_t* proofs, const RaggedGt* ent, size_t npow, size_t nz, const uint64_t* challenges, uint32_t* factors, cudaStream_t s) {
    const size_t blocks = (2 * npow + SIPP_ACCUM_GROUPS - 1) / SIPP_ACCUM_GROUPS + (6 * nz + SIPP_ACCUM_THREADS - 1) / SIPP_ACCUM_THREADS;
    if (blocks == 0) return 0;
    k_gt_fold_ragged<<<(unsigned)blocks, SIPP_ACCUM_THREADS, 0, s>>>(proofs, ent, npow, nz, challenges, factors);
    return (int)cudaGetLastError();
}
int launch_qlines_batch(const uint32_t* B, size_t npoints, uint32_t* qlines, cudaStream_t s) {
    k_qlines_batch<<<(unsigned)((npoints + 63) / 64), 64, 0, s>>>(B, npoints, qlines);
    return (int)cudaGetLastError();
}
int launch_eval_lines_batch(const uint32_t* A, const uint32_t* B, const BatchJob& job, size_t p0, size_t np, const uint32_t* qlines, uint32_t* lines,
                            cudaStream_t s) {
    size_t threads = np * job.h * SIPP_LINES_PER_PAIR;
    k_eval_lines_batch<<<(unsigned)((threads + 127) / 128), 128, 0, s>>>(A, B, job, p0, np, qlines, lines);
    return (int)cudaGetLastError();
}
int launch_eval_lines_mat(const uint32_t* A, const uint32_t* B, size_t nr, size_t m, const uint32_t* qlines, uint32_t* lines, cudaStream_t s) {
    const size_t threads = nr * nr * m * SIPP_LINES_PER_PAIR;
    k_eval_lines_mat<<<(unsigned)((threads + 127) / 128), 128, 0, s>>>(A, B, nr, m, qlines, lines);
    return (int)cudaGetLastError();
}
size_t qlines_bytes_per_point() { return (size_t)SIPP_LINES_PER_PAIR * SIPP_QLINE_WORDS * sizeof(uint32_t); }
size_t lines_bytes_per_pair() { return (size_t)SIPP_PAIR_LINE_WORDS * sizeof(uint32_t); }

}  // namespace sipp

// k_products.cu -- kernels of the batched independent products (products.cu: sipp_inner_product_batch and friends).
//
//   k_accum_plan    k_accum's 6-lane accumulation over the line table of one chunk, but every group reads its pair range
//                   (first pair, pair count) from the host plan instead of gid * kpg, so groups follow the segments of a ragged
//                   batch.  One un-exponentiated partial per group, at partials[global group id].
//   k_seg_product   one pass of the segmented product: every block multiplies a run of at most SIPP_PRODUCT_SPAN consecutive
//                   Fq12 of one segment (2 per 6-lane group, then the block tree) into one.  The host chains passes until every
//                   segment is one element, so the depth is logarithmic in the longest segment.  An empty run gives 1.
//   k_ragged_gather / k_scatter_fq12   the per-round gather and the proof-slot scatter of the ragged batched prover
//   k_gather_points  the final points of the ragged batched verifier
#include "accum.cuh"
#include "device_common.cuh"

namespace sipp {

__global__ void __launch_bounds__(SIPP_ACCUM_THREADS, SIPP_ACCUM_MINBLOCKS) k_accum_plan(const uint32_t* __restrict__ lines, const ProductGroup* __restrict__ plan,
                                                                                   size_t g0, size_t ngroups, size_t c0, int kpg,
                                                                                   uint32_t* __restrict__ partials) {
    __shared__ __align__(16) uint32_t stage[SIPP_ACCUM_GROUPS][2][SIPP_LINE_WORDS];
    const Lane6 L = lane6_of_thread();
    const int warp = threadIdx.x >> 5;
    const int group = warp * SIPP_GROUPS_PER_WARP + L.base / 6;
    const bool active_lane = L.k < 6;
    const int grp = active_lane ? group : warp * SIPP_GROUPS_PER_WARP;  // idle lanes shadow group 0 of the warp (results unused)
    const int k = active_lane ? L.k : 0;
    const size_t gid = (size_t)blockIdx.x * SIPP_ACCUM_GROUPS + grp;
    const ProductGroup pg = gid < ngroups ? plan[g0 + gid] : ProductGroup{(uint32_t)c0, 0};
    const int npairs = (int)pg.pairs;
    const uint32_t* base = lines + ((size_t)pg.first - c0) * SIPP_PAIR_LINE_WORDS;

    // the rest is k_accum's schedule: step-major line fetches (step s, pair q), staged one line ahead with cp.async
    const int total = SIPP_LINES_PER_PAIR * npairs;
    auto line_ptr = [&](int idx) { int s = idx / (npairs > 0 ? npairs : 1); int q = idx - s * (npairs > 0 ? npairs : 1);
                                   return base + (size_t)q * SIPP_PAIR_LINE_WORDS + s * SIPP_LINE_WORDS; };
    auto prefetch = [&](int idx, int buf) {
        if (active_lane && idx < total) {
            const uint32_t* src = line_ptr(idx);
            for (int c = k; c < 20; c += 6) cp_async16(&stage[grp][buf][c * 4], src + c * 4);
        }
        cp_async_commit();
    };

    Fq2 f = lane_one(k);
    int fetch = 0;
    prefetch(0, 0);
    const unsigned long long plus = SIPP_ATE_PLUS_MASK, minus = SIPP_ATE_MINUS_MASK;
    // uniform control flow over kpg steps per line (shuffles inside); a group with fewer pairs multiplies by stale data it discards
    const int maxpairs = kpg;
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
    if (active_lane && npairs > 0) store_fq2_words(partials + (g0 + gid) * 96 + k * 16, f);
}

#define SIPP_PRODUCT_PER_GROUP 2
static_assert(SIPP_PRODUCT_SPAN == SIPP_ACCUM_GROUPS * SIPP_PRODUCT_PER_GROUP, "launch.h SIPP_PRODUCT_SPAN");

// one block per task: work[dst] = prod_{i < n} work[src + i]  (n <= SIPP_PRODUCT_SPAN; n = 0 gives 1)
__global__ void __launch_bounds__(SIPP_ACCUM_THREADS) k_seg_product(const ProductTask* __restrict__ tasks, uint32_t* __restrict__ work) {
    __shared__ __align__(16) uint32_t red[SIPP_ACCUM_GROUPS * 96];
    const Lane6 L = lane6_of_thread();
    const int warp = threadIdx.x >> 5;
    const bool active_lane = L.k < 6;
    const int group = active_lane ? warp * SIPP_GROUPS_PER_WARP + L.base / 6 : SIPP_ACCUM_GROUPS;
    const int k = active_lane ? L.k : 0;
    const ProductTask t = tasks[blockIdx.x];
    const int n = (int)t.n;
    Fq2 f = lane_one(k);
    const int rounds = (n + SIPP_ACCUM_GROUPS - 1) / SIPP_ACCUM_GROUPS;  // block-uniform
    for (int r = 0; r < rounds; r++) {
        const int i = r * SIPP_ACCUM_GROUPS + group;
        const bool have = active_lane && i < n;
        const Fq2 v = have ? load_fq2_words(work + ((size_t)t.src + i) * 96 + k * 16) : lane_one(k);
        f = r == 0 ? v : coop_mul(L, f, v);
    }
    const int live = n < SIPP_ACCUM_GROUPS ? n : SIPP_ACCUM_GROUPS;
    if (live > 1) f = block_product_coop(L, f, red, group, live);
    if (active_lane && group == 0) store_fq2_words(work + (size_t)t.dst * 96 + k * 16, f);
}

// ragged batched prover (ragged.cu), rounds >= 1: per active instance (h = current n / 2), gA / gB <- A_hi || A_lo and B_lo || B_hi
// at pairs [2 estart, 2 estart + 2h), so that Z_L = <A_hi, B_lo> (prover_native.rs:48) and Z_R = <A_lo, B_hi> (:49) are two
// consecutive segments of the products path.  One thread per 16-byte quarter of a Montgomery point: 4 of A_hi, 4 of A_lo, 8 of
// B_lo, 8 of B_hi per element.
#define SIPP_GATHER_QUADS 24
__global__ void __launch_bounds__(256) k_ragged_gather(const uint32_t* __restrict__ A, const uint32_t* __restrict__ B, const RaggedInst* __restrict__ tab,
                                                       unsigned act, size_t elems, uint32_t* __restrict__ gA, uint32_t* __restrict__ gB) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= elems * SIPP_GATHER_QUADS) return;
    const size_t e = t / SIPP_GATHER_QUADS;
    const int q = (int)(t % SIPP_GATHER_QUADS);
    unsigned lo = 0, hi = act - 1;  // last instance whose elements start at or before e
    while (lo < hi) {
        const unsigned mid = (lo + hi + 1) >> 1;
        if ((size_t)tab[mid].estart <= e) lo = mid; else hi = mid - 1;
    }
    const RaggedInst r = tab[lo];
    const size_t i = e - r.estart, src_lo = (size_t)r.base + i, src_hi = src_lo + r.h;
    const size_t dst_l = 2 * (size_t)r.estart + i, dst_r = dst_l + r.h;  // Z_L segment, Z_R segment
    const uint4* sA = reinterpret_cast<const uint4*>(A);
    const uint4* sB = reinterpret_cast<const uint4*>(B);
    uint4* dA = reinterpret_cast<uint4*>(gA);
    uint4* dB = reinterpret_cast<uint4*>(gB);
    if (q < 4) dA[4 * dst_l + q] = sA[4 * src_hi + q];
    else if (q < 8) dA[4 * dst_r + q - 4] = sA[4 * src_lo + q - 4];
    else if (q < 16) dB[8 * dst_l + q - 8] = sB[8 * src_lo + q - 8];
    else dB[8 * dst_r + q - 16] = sB[8 * src_hi + q - 16];
}

// proofs[dst[j]] <- res[j]: the products of a round into the proof slots of their instances, 24 quarters of an Fq12 per thread row
__global__ void __launch_bounds__(256) k_scatter_fq12(const uint32_t* __restrict__ res, const uint64_t* __restrict__ dst, size_t count,
                                                      uint32_t* __restrict__ proofs) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= count * 24) return;
    const size_t j = t / 24, q = t % 24;
    reinterpret_cast<uint4*>(proofs)[24 * dst[j] + q] = reinterpret_cast<const uint4*>(res)[24 * j + q];
}

// ragged batched verifier (ragged.cu): the final A, B of every instance -- its first point once every fold has run
// (verifier_native.rs:74-75) -- side by side for the final pairings: gA[j] <- A[at[j]], gB[j] <- B[at[j]].  One thread per 16-byte
// quarter of a Montgomery point: 4 of A, 8 of B per instance.
__global__ void __launch_bounds__(256) k_gather_points(const uint32_t* __restrict__ A, const uint32_t* __restrict__ B, const uint64_t* __restrict__ at,
                                                       size_t count, uint32_t* __restrict__ gA, uint32_t* __restrict__ gB) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= count * 12) return;
    const size_t j = t / 12, src = at[j];
    const int q = (int)(t % 12);
    if (q < 4) reinterpret_cast<uint4*>(gA)[4 * j + q] = reinterpret_cast<const uint4*>(A)[4 * src + q];
    else reinterpret_cast<uint4*>(gB)[8 * j + q - 4] = reinterpret_cast<const uint4*>(B)[8 * src + q - 4];
}

// ------------------------------------------------------------------------------------------------ launch wrappers
int launch_ragged_gather(const uint32_t* A, const uint32_t* B, const RaggedInst* tab, unsigned act, size_t elems, uint32_t* gA, uint32_t* gB, cudaStream_t s) {
    const size_t threads = elems * SIPP_GATHER_QUADS;
    k_ragged_gather<<<(unsigned)((threads + 255) / 256), 256, 0, s>>>(A, B, tab, act, elems, gA, gB);
    return (int)cudaGetLastError();
}
int launch_scatter_fq12(const uint32_t* res, const uint64_t* dst, size_t count, uint32_t* proofs, cudaStream_t s) {
    k_scatter_fq12<<<(unsigned)((count * 24 + 255) / 256), 256, 0, s>>>(res, dst, count, proofs);
    return (int)cudaGetLastError();
}
int launch_gather_points(const uint32_t* A, const uint32_t* B, const uint64_t* at, size_t count, uint32_t* gA, uint32_t* gB, cudaStream_t s) {
    k_gather_points<<<(unsigned)((count * 12 + 255) / 256), 256, 0, s>>>(A, B, at, count, gA, gB);
    return (int)cudaGetLastError();
}
int launch_accum_plan(const uint32_t* lines, const ProductGroup* plan, size_t g0, size_t ngroups, size_t c0, int kpg, uint32_t* partials, cudaStream_t s) {
    const size_t blocks = (ngroups + SIPP_ACCUM_GROUPS - 1) / SIPP_ACCUM_GROUPS;
    k_accum_plan<<<(unsigned)blocks, SIPP_ACCUM_THREADS, 0, s>>>(lines, plan, g0, ngroups, c0, kpg, partials);
    return (int)cudaGetLastError();
}
int launch_seg_product(const ProductTask* tasks, size_t ntasks, uint32_t* work, cudaStream_t s) {
    k_seg_product<<<(unsigned)ntasks, SIPP_ACCUM_THREADS, 0, s>>>(tasks, work);
    return (int)cudaGetLastError();
}

}  // namespace sipp

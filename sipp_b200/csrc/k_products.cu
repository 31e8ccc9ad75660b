// k_products.cu -- kernels of the batched independent products (products.cu: sipp_inner_product_batch and friends).
//
//   k_accum_plan    k_accum's 6-lane accumulation over the line table of one chunk, but every group reads its pair range
//                   (first pair, pair count) from the host plan instead of gid * kpg, so groups follow the segments of a ragged
//                   batch.  One un-exponentiated partial per group, at partials[global group id].
//   k_seg_product   one pass of the segmented product: every block multiplies a run of at most SIPP_PRODUCT_SPAN consecutive
//                   Fq12 of one segment (2 per 6-lane group, then the block tree) into one.  The host chains passes until every
//                   segment is one element, so the depth is logarithmic in the longest segment.  An empty run gives 1.
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

// ------------------------------------------------------------------------------------------------ launch wrappers
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

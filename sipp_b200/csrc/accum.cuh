// accum.cuh -- pieces of the 6-lane line accumulation shared by k_accum (k_coop.cu) and k_accum_plan (k_products.cu): the
// line-table layout, the block shape, cp.async staging and the block-level tree product of the groups' accumulators.
#pragma once
#include "coop.cuh"

namespace sipp {

#define SIPP_LINE_WORDS 80                               // 5 Fq2
#define SIPP_PAIR_LINE_WORDS (SIPP_LINES_PER_PAIR * SIPP_LINE_WORDS)
#ifndef SIPP_ACCUM_THREADS
#define SIPP_ACCUM_THREADS 128
#endif
#define SIPP_GROUPS_PER_WARP 5
#define SIPP_ACCUM_GROUPS (SIPP_ACCUM_THREADS / 32 * SIPP_GROUPS_PER_WARP)
#ifndef SIPP_ACCUM_MINBLOCKS
#define SIPP_ACCUM_MINBLOCKS 2
#endif

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

__device__ __forceinline__ Fq2 lane_one(int k) { return k == 0 ? fq2_one() : fq2_zero(); }

// tree product over the groups of a block; result in group 0.  sh: [groups][96 words]
static __device__ __noinline__ Fq2 block_product_coop(const Lane6& L, Fq2 f, uint32_t* sh, int group, int ngroups) {
    const int k = L.k < 6 ? L.k : 0;
    int n = ngroups;
    while (n > 1) {
        int half = (n + 1) >> 1;
        __syncthreads();
        if (L.k < 6 && group >= half && group < n) store_fq2_words(sh + group * 96 + k * 16, f);
        __syncthreads();
        bool take = group + half < n;
        Fq2 other = take ? load_fq2_words(sh + (group + half) * 96 + k * 16) : lane_one(k);
        f = coop_mul(L, f, other);
        n = half;
    }
    return f;
}

}  // namespace sipp

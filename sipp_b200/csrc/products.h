// products.h -- the batched independent products path (products.cu), shared by sipp_inner_product_batch and the ragged batched
// prover (ragged.cu): a host plan of accumulator groups and segment-product tasks, then one launch sequence over decoded points.
#pragma once
#include <stddef.h>

#include <vector>

#include "host_state.h"

namespace sipp_host {

// line-table budget of one call: the same as a batched proof's (batch.cu)
const size_t kProductLinesCap = (size_t)16 << 30;

struct ProductPlan {
    int kpg = 1;
    size_t chunk_pairs = 0;                 // pairs per chunk (the last one may be shorter)
    std::vector<sipp::ProductGroup> groups; // in pair order: segment by segment, chunk by chunk
    std::vector<size_t> seg_first_group;    // count + 1 entries: the groups of segment j are [seg_first_group[j], seg_first_group[j + 1])
    std::vector<size_t> chunk_first_group;  // chunks + 1 entries
    // k_seg_product passes over the work array [group partials | intermediate runs | one product per segment]
    std::vector<sipp::ProductTask> tasks;
    std::vector<size_t> pass_first;
    size_t seg0 = 0;                        // work slot of segment 0's product (the products are consecutive)
    size_t chunks() const { return chunk_first_group.size() - 1; }
    size_t work_slots(size_t count) const { return seg0 + count; }
};

// offsets: count + 1 checked CSR offsets; fills the groups and the tasks
int product_plan(const size_t* offsets, size_t count, int kpg_max, size_t chunk_pairs, ProductPlan& p);
// lines -> accumulation -> segment products -> final exponentiation of the `count` products of n decoded pairs (dA, dB, Montgomery)
// into res[count][96 words] (boundary bytes).  dgroups / dtasks: the plan's groups and tasks on the device; work: plan.work_slots(count)
// Fq12; the line table must already hold min(n, plan.chunk_pairs) pairs.  Enqueues on s.
int products_launch(const uint32_t* dA, const uint32_t* dB, size_t n, size_t count, const ProductPlan& plan, const sipp::ProductGroup* dgroups,
                    const sipp::ProductTask* dtasks, uint32_t* work, uint32_t* res, cudaStream_t s);

}  // namespace sipp_host

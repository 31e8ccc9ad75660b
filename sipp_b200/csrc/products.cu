// products.cu -- batched independent products (C ABI: sipp_inner_product_batch, sipp_inner_product_batch_device,
// sipp_pairing_batch).
//
// `count` products of arbitrary, unequal lengths in one launch set: out[j] = prod_{offsets[j] <= i < offsets[j+1]} e(A_i, B_i), each
// exactly sipp_inner_product (prover_native.rs:15-23) on its segment.  One call pays the fixed costs (upload, decode, validation,
// the latency floors of lines, accumulation and final exponentiation, one synchronisation) once for all products:
//   plan (host)      every segment is cut into accumulator groups of at most kpg consecutive pairs; no group crosses a segment
//                    or a chunk (a run of pairs whose line table fits the budget)
//   lines            k_lines / k_lines_wide on the flat pair list, one chunk at a time
//   accumulation     k_accum_plan: one partial per group
//   segmented product k_seg_product passes: one un-exponentiated Fq12 per segment, depth logarithmic in the longest segment
//   final exp.       k_fe_batch_eng / k_fe_batch, one per segment, boundary bytes
#include <vector>

#include "products.h"

using namespace sipp;
using namespace sipp_host;

namespace {
void product_tasks(ProductPlan& p, size_t count);
}  // namespace

namespace sipp_host {

// offsets already checked (products_args)
int product_plan(const size_t* offsets, size_t count, int kpg_max, size_t chunk_pairs, ProductPlan& p) {
    const size_t total = offsets[count];
    if (total > (size_t)UINT32_MAX) return fail(SIPP_ERR_ARG, "inner_product_batch: more than 2^32 - 1 pairs");
    size_t longest = 0;
    for (size_t j = 0; j < count; j++)
        if (offsets[j + 1] - offsets[j] > longest) longest = offsets[j + 1] - offsets[j];
    // kpg pairs of one segment share an accumulator and its 64 squarings (5,070 Fq-mul-eq per group, 3,661 per pair; the kernel runs
    // kpg steps whatever the group holds).  The GPU holds 2 blocks x 20 groups per SM at a time: the kpg that minimises waves x group
    // length, the cost model of batched proofs (batch.cu: batch_products) with the group count of the actual segments.  Any integer:
    // one segment of 2^16 pairs takes kpg = 12, one wave, like sipp_inner_product, where the powers of two would need 3 waves of 4.
    p.kpg = 1;
    {
        const size_t wave = (size_t)g_sm_count * 40;
        double best = 0;
        for (size_t cand = 1; cand <= (size_t)(kpg_max < 1 ? 1 : kpg_max) && cand <= (longest ? longest : 1); cand++) {
            size_t groups = 0;
            for (size_t j = 0; j < count; j++) groups += (offsets[j + 1] - offsets[j] + cand - 1) / cand;
            double cost = (double)((groups + wave - 1) / wave) * (5070.0 + 3661.0 * (double)cand);
            if (best == 0 || cost < best) { best = cost; p.kpg = (int)cand; }
            if (groups <= wave) break;  // one wave: a longer group only costs more
        }
    }
    const size_t budget = kProductLinesCap / lines_bytes_per_pair();
    p.chunk_pairs = chunk_pairs ? (chunk_pairs < budget ? chunk_pairs : budget) : budget;
    p.groups.clear();
    p.seg_first_group.assign(count + 1, 0);
    p.chunk_first_group.clear();
    for (size_t j = 0; j < count; j++) {
        p.seg_first_group[j] = p.groups.size();
        for (size_t q = offsets[j]; q < offsets[j + 1];) {
            const size_t chunk = q / p.chunk_pairs;
            if (chunk == p.chunk_first_group.size()) p.chunk_first_group.push_back(p.groups.size());
            size_t e = q + (size_t)p.kpg;
            if (e > offsets[j + 1]) e = offsets[j + 1];
            if (e > (chunk + 1) * p.chunk_pairs) e = (chunk + 1) * p.chunk_pairs;
            p.groups.push_back(ProductGroup{(uint32_t)q, (uint32_t)(e - q)});
            q = e;
        }
    }
    p.seg_first_group[count] = p.groups.size();
    p.chunk_first_group.push_back(p.groups.size());
    product_tasks(p, count);
    return SIPP_OK;
}

int products_launch(const uint32_t* dA, const uint32_t* dB, size_t n, size_t count, const ProductPlan& plan, const ProductGroup* dgroups,
                    const ProductTask* dtasks, uint32_t* work, uint32_t* res, cudaStream_t s) {
    {
        Span sp(0, s);
        MillerJob job;
        job.a_off[0] = job.b_off[0] = job.a_off[1] = job.b_off[1] = 0;
        job.m = n;
        for (size_t c = 0; c < plan.chunks(); c++) {
            const size_t c0 = c * plan.chunk_pairs, cur = n - c0 < plan.chunk_pairs ? n - c0 : plan.chunk_pairs;
            const size_t g0 = plan.chunk_first_group[c], ng = plan.chunk_first_group[c + 1] - g0;
            uint32_t* lines = lines_buffer();
            // 16 lanes per pair for a launch that cannot fill the GPU, one thread per pair otherwise (as ctx_products_to_device)
            const bool wide = cur <= (size_t)g_opt_wide_max;
            int le = wide ? launch_lines_wide(dA, dB, job, 1, c0, cur, lines, s) : launch_lines(dA, dB, job, 1, c0, cur, lines, s);
            if (le) return cuda_fail((cudaError_t)le, "k_lines");
            le = launch_accum_plan(lines, dgroups, g0, ng, c0, plan.kpg, work, s);
            if (le) return cuda_fail((cudaError_t)le, "k_accum_plan");
            g_stats.launches += 2;
            g_stats.miller_launches++;
        }
    }
    g_stats.miller_pairs += n;
    {
        Span sp(1, s);
        for (size_t k = 0; k + 1 < plan.pass_first.size(); k++) {
            int le = launch_seg_product(dtasks + plan.pass_first[k], plan.pass_first[k + 1] - plan.pass_first[k], work, s);
            if (le) return cuda_fail((cudaError_t)le, "k_seg_product");
            g_stats.launches++;
        }
        // one 32-lane machine per product while they all fit the GPU at once, 6-lane groups beyond (as batch_products)
        const uint32_t* seg = work + plan.seg0 * 96;
        int le = (g_opt_fe_engine && count <= (size_t)g_sm_count * 12) ? launch_fe_batch_eng(seg, count, 1, 1, res, 96, 0, 0, g_opt_fe_norm, s)
                                                                       : launch_fe_batch(seg, count, 1, 1, res, 96, 0, 0, g_opt_fe_norm, s);
        if (le) return cuda_fail((cudaError_t)le, "k_fe_batch");
        g_stats.launches++;
    }
    return SIPP_OK;
}

}  // namespace sipp_host

namespace {

// passes of k_seg_product over the work array [group partials | intermediate runs | one product per segment]; p.seg0 = the slot
// of segment 0's product (the `count` products are consecutive)
void product_tasks(ProductPlan& p, size_t count) {
    std::vector<ProductTask>& tasks = p.tasks;
    std::vector<size_t>& pass_first = p.pass_first;
    std::vector<size_t> start(count), len(count);
    size_t longest = 0;
    for (size_t j = 0; j < count; j++) {
        start[j] = p.seg_first_group[j];
        len[j] = p.seg_first_group[j + 1] - start[j];
        if (len[j] > longest) longest = len[j];
    }
    size_t next = p.groups.size();
    tasks.clear();
    pass_first.clear();
    // segments longer than one task shrink SIPP_PRODUCT_SPAN-fold per pass; the others wait where they are
    while (longest > SIPP_PRODUCT_SPAN) {
        pass_first.push_back(tasks.size());
        longest = 0;
        for (size_t j = 0; j < count; j++) {
            if (len[j] <= SIPP_PRODUCT_SPAN) continue;
            const size_t nb = (len[j] + SIPP_PRODUCT_SPAN - 1) / SIPP_PRODUCT_SPAN;
            for (size_t b = 0; b < nb; b++) {
                const size_t n = len[j] - b * SIPP_PRODUCT_SPAN < SIPP_PRODUCT_SPAN ? len[j] - b * SIPP_PRODUCT_SPAN : SIPP_PRODUCT_SPAN;
                tasks.push_back(ProductTask{(uint32_t)(start[j] + b * SIPP_PRODUCT_SPAN), (uint32_t)n, (uint32_t)(next + b), 0});
            }
            start[j] = next;
            len[j] = nb;
            next += nb;
            if (nb > longest) longest = nb;
        }
    }
    // last pass: every segment, empty ones included (n = 0 writes 1)
    pass_first.push_back(tasks.size());
    for (size_t j = 0; j < count; j++) tasks.push_back(ProductTask{(uint32_t)start[j], (uint32_t)len[j], (uint32_t)(next + j), 0});
    pass_first.push_back(tasks.size());
    p.seg0 = next;
}

int products_args(const void* A, size_t a_len, const void* B, size_t b_len, const size_t* offsets, size_t count, const void* out) {
    if (a_len != b_len) return fail(SIPP_ERR_LENGTH, "assert_eq!(A.len(), B.len())");
    if (count == 0) return a_len == 0 ? SIPP_OK : fail(SIPP_ERR_ARG, "inner_product_batch: count == 0 with pairs");
    if (!A || !B || !offsets || !out) return fail(SIPP_ERR_ARG, "inner_product_batch: null pointer");
    if (offsets[0] != 0) return fail(SIPP_ERR_ARG, "inner_product_batch: offsets[0] != 0");
    for (size_t j = 0; j < count; j++)
        if (offsets[j + 1] < offsets[j]) return fail(SIPP_ERR_ARG, "inner_product_batch: decreasing offsets");
    if (offsets[count] != a_len) return fail(SIPP_ERR_ARG, "inner_product_batch: offsets[count] != number of pairs");
    return SIPP_OK;
}

// the whole call on the device: bytesA / bytesB hold the boundary bytes (the caller's buffers or staging copies); the products
// (boundary bytes) are copied to `out` (host or device memory, per out_kind) only when every point passed its checks
int products_run(const uint32_t* bytesA, const uint32_t* bytesB, size_t n, const size_t* offsets, size_t count, void* out, cudaMemcpyKind out_kind) {
    cudaStream_t s = g_stream;
    ProductPlan plan;
    int rc = product_plan(offsets, count, g_opt_batch_kpg_max, (size_t)g_opt_product_chunk, plan);
    if (rc) return rc;
    const std::vector<ProductTask>& tasks = plan.tasks;
    const size_t slots = plan.work_slots(count);
    uint32_t *dA = nullptr, *dB = nullptr, *work = nullptr, *res = nullptr;
    ProductGroup* dgroups = nullptr;
    ProductTask* dtasks = nullptr;
    int* flags = nullptr;
    cudaError_t e = pool_alloc((void**)&dA, n * 64);
    if (e == cudaSuccess) e = pool_alloc((void**)&dB, n * 128);
    if (e == cudaSuccess) e = pool_alloc((void**)&work, slots * 384);
    if (e == cudaSuccess) e = pool_alloc((void**)&res, count * 384);
    if (e == cudaSuccess) e = pool_alloc((void**)&dgroups, plan.groups.size() * sizeof(ProductGroup));
    if (e == cudaSuccess) e = pool_alloc((void**)&dtasks, tasks.size() * sizeof(ProductTask));
    if (e == cudaSuccess) e = pool_alloc((void**)&flags, sizeof(int));
    struct Release {
        std::vector<void*> p;
        ~Release() { for (void* q : p) pool_free(q); }
    } release{{dA, dB, work, res, dgroups, dtasks, flags}};  // recycled blocks: later work on the same stream only
    if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(inner_product_batch)");
    auto run = [&]() -> int {
        CK(cudaMemsetAsync(flags, 0, sizeof(int), s));
        if (!plan.groups.empty()) CK(cudaMemcpyAsync(dgroups, plan.groups.data(), plan.groups.size() * sizeof(ProductGroup), cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(dtasks, tasks.data(), tasks.size() * sizeof(ProductTask), cudaMemcpyHostToDevice, s));
        if (n) {
            Span sp(3, s);
            int le = launch_codec_decode(bytesA, dA, n * 2, flags, s);
            if (!le) le = launch_codec_decode(bytesB, dB, n * 4, flags, s);
            if (le) return cuda_fail((cudaError_t)le, "k_codec_decode");
            g_stats.launches += 2;
            if (g_opt_validate) {  // on the curve, B_i in the order-r subgroup (SIPP_OPT_VALIDATE_POINTS), as sipp_inner_product
                le = launch_validate_points(dA, dB, n, flags, s);
                if (le) return cuda_fail((cudaError_t)le, "k_validate_points");
                g_stats.launches++;
            }
        }
        if (plan.chunks()) {
            const int lr = lines_reserve((n < plan.chunk_pairs ? n : plan.chunk_pairs) * lines_bytes_per_pair());
            if (lr) return lr;
        }
        const int pr = products_launch(dA, dB, n, count, plan, dgroups, dtasks, work, res, s);
        if (pr) return pr;
        int flag = 0;
        CK(cudaMemcpyAsync(&flag, flags, sizeof(int), cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        if (flag & 1) return fail(SIPP_ERR_ENCODING, "input coordinate >= p");
        if (flag & 2) return fail(SIPP_ERR_ENCODING, "input point is not on the curve");
        if (flag & 4) return fail(SIPP_ERR_ENCODING, "input G2 point is not in the prime-order subgroup");
        CK(cudaMemcpyAsync(out, res, count * 384, out_kind, s));
        CK(cudaStreamSynchronize(s));
        return SIPP_OK;
    };
    rc = run();
    if (rc) cudaStreamSynchronize(s);
    return rc;
}

}  // namespace

extern "C" {

int sipp_inner_product_batch(const uint8_t* A, size_t a_len, const uint8_t* B, size_t b_len, const size_t* offsets, size_t count, uint8_t* out) {
    int rc = products_args(A, a_len, B, b_len, offsets, count, out);
    if (rc || count == 0) return rc ? rc : ensure_init();
    rc = ensure_init();
    if (rc) return rc;
    uint32_t *tA = nullptr, *tB = nullptr;
    cudaError_t e = pool_alloc((void**)&tA, a_len * 64);
    if (e == cudaSuccess) e = pool_alloc((void**)&tB, a_len * 128);
    struct Release {
        uint32_t *a, *b;
        ~Release() { pool_free(a); pool_free(b); }
    } release{tA, tB};
    if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(inner_product_batch)");
    if (a_len) {
        CK(cudaMemcpyAsync(tA, A, a_len * 64, cudaMemcpyHostToDevice, g_stream));
        CK(cudaMemcpyAsync(tB, B, a_len * 128, cudaMemcpyHostToDevice, g_stream));
    }
    return products_run(tA, tB, a_len, offsets, count, out, cudaMemcpyDeviceToHost);  // synchronises: the staging blocks are idle on return
}

int sipp_inner_product_batch_device(const void* dA, const void* dB, size_t n, const size_t* offsets, size_t count, void* d_out) {
    int rc = products_args(dA, n, dB, n, offsets, count, d_out);
    if (rc || count == 0) return rc ? rc : ensure_init();
    rc = ensure_init();
    if (rc) return rc;
    return products_run((const uint32_t*)dA, (const uint32_t*)dB, n, offsets, count, d_out, cudaMemcpyDeviceToDevice);
}

int sipp_pairing_batch(const uint8_t* a, const uint8_t* b, size_t count, uint8_t* out) {
    std::vector<size_t> offsets(count + 1);
    for (size_t j = 0; j <= count; j++) offsets[j] = j;
    return sipp_inner_product_batch(a, count, b, count, offsets.data(), count, out);
}

// host-only plan of a batch (no GPU needed): 4 words (first pair, pairs, segment, chunk) per accumulator group to `out` when
// out_cap >= 4 x groups, kpg to *kpg_out; returns the number of groups or a negative status
long sipp_test_product_plan(const size_t* offsets, size_t count, int kpg_max, size_t chunk_pairs, size_t* out, size_t out_cap, int* kpg_out) {
    if (!offsets) return fail(SIPP_ERR_ARG, "null offsets");
    if (count == 0) return 0;
    const size_t n = offsets[count];
    int rc = products_args(offsets, n, offsets, n, offsets, count, offsets);  // the offsets checks of the entry points
    if (rc) return rc;
    ProductPlan plan;
    rc = product_plan(offsets, count, kpg_max, chunk_pairs, plan);
    if (rc) return rc;
    if (kpg_out) *kpg_out = plan.kpg;
    const size_t g = plan.groups.size();
    if (out && out_cap >= 4 * g) {
        size_t seg = 0;
        for (size_t i = 0; i < g; i++) {
            while (plan.seg_first_group[seg + 1] <= i) seg++;
            out[4 * i] = plan.groups[i].first;
            out[4 * i + 1] = plan.groups[i].pairs;
            out[4 * i + 2] = seg;
            out[4 * i + 3] = plan.groups[i].first / plan.chunk_pairs;
        }
    }
    return (long)g;
}

}  // extern "C"

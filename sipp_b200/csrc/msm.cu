// msm.cu -- batched multi-scalar multiplications (C ABI: sipp_g1_msm_batch, sipp_g2_msm_batch and their _device forms; test hook
// sipp_test_msm_plan) and batched multi-exponentiations in Fq12 (sipp_gt_msm_batch and its _device form; test hook
// sipp_test_gt_msm_plan).  Kernels: k_msm.cu, k_gt_msm.cu; recoding and bucket arithmetic: msm.cuh.
//
// `count` independent MSMs of unequal lengths in one call: out[j] = sum_{offsets[j] <= i < offsets[j+1]} [k_i] P_i.  Every segment is
// planned on the host from its length alone:
//   Straus     (1 <= len < SIPP_MSM_STRAUS_BELOW_G1 / _G2): one thread per segment, shared doublings over the NAF digits of its terms
//   Pippenger  (from there on): signed c-bit windows, c from the cost model msm_window_bits; the buckets of all
//              Pippenger segments are filled by one sort of (bucket, term) entries
// Empty segments take the Straus path with no terms and give the identity.
//
// The GT multi-exponentiation (group 3 below) is planned the same way: out[j] = prod g_i^(k_i) in Fq12, each segment either on the short
// path (len < SIPP_GT_MSM_SHORT_BELOW: one generic power per element, k_gt_msm_pow, then k_seg_product) or on Pippenger with unsigned
// c-bit windows (k_gt_msm.cu), whose results join the segmented product as one factor each.
#include <string.h>

#include <vector>

#include "host_state.h"
#include "products.h"

using namespace sipp;
using namespace sipp_host;

// Segments shorter than this take the Straus path: where the two paths, both timed at every length (sipp_test_msm_batch_device), cross
// for 4,096 segments on one B200 (tools/msm_time.py, DESIGN §7) -- G1 at 13 points, G2 at 8.
#define SIPP_MSM_STRAUS_BELOW_G1 13
#define SIPP_MSM_STRAUS_BELOW_G2 8
#define SIPP_MSM_MIN_C 5
#define SIPP_MSM_MAX_C 16
#define SIPP_MSM_BUCKETS_PER_THREAD 8  // k_msm_windows: running sums of at most 8 buckets per thread, 64 threads per block
// GT segments shorter than this take the short path: where the two paths, both forced (sipp_test_gt_msm_batch_device), cross for batches
// of many segments on one B200 (tools/gt_msm_time.py, DESIGN §7: 4,096 x 256 elements, short path faster; 2,048 x 512, Pippenger
// faster).  One segment alone crosses later, between 2^12 and 2^14 elements.
#define SIPP_GT_MSM_SHORT_BELOW 512
#define SIPP_GT_MSM_MIN_C 2

namespace {

// group 1 = G1, 2 = G2, 3 = GT (the multi-exponentiation in Fq12)
struct GroupInfo {
    int nc, bits, words;  // sub-scalars per scalar, bound of a sub-scalar, u32 words of an input element
    bool gt;              // unsigned digits: ceil(bits / c) windows of 2^c - 1 buckets (signed: bits / c + 1 windows of 2^(c-1))
};
GroupInfo group_info(int group) { return group == 1 ? GroupInfo{2, 128, 16, false} : group == 2 ? GroupInfo{4, 66, 32, false} : GroupInfo{1, 254, 96, true}; }

int windows_of(const GroupInfo& g, int c) { return g.gt ? (g.bits + c - 1) / c : g.bits / c + 1; }
size_t buckets_of(const GroupInfo& g, int c) { return g.gt ? ((size_t)1 << c) - 1 : (size_t)1 << (c - 1); }

// the window size of a Pippenger segment.  G1 / G2: the c minimising W (NC len + 3 2^(c-1)) -- one mixed addition per term and window
// to fill the buckets, two Jacobian additions (about 1.5 mixed ones each) per bucket to reduce them.  GT: W (len + 2 2^c) + c W Fq12
// products -- one per element and window, two per bucket, c squarings per window.
int msm_window_bits(int group, size_t len) {
    const GroupInfo g = group_info(group);
    const int lo = g.gt ? SIPP_GT_MSM_MIN_C : SIPP_MSM_MIN_C;
    int best = lo;
    double best_cost = 0;
    for (int c = lo; c <= SIPP_MSM_MAX_C; c++) {
        const double W = windows_of(g, c);
        const double cost = g.gt ? W * ((double)len + 2.0 * (double)(1u << c)) + c * W
                                 : W * ((double)g.nc * (double)len + 3.0 * (double)(1u << (c - 1)));
        if (c == lo || cost < best_cost) {
            best_cost = cost;
            best = c;
        }
    }
    return best;
}

// 0: Straus (the short path in GT), else the window bits of the Pippenger path
int msm_segment_c(int group, size_t len) {
    const size_t below = group == 1 ? SIPP_MSM_STRAUS_BELOW_G1 : group == 2 ? SIPP_MSM_STRAUS_BELOW_G2 : SIPP_GT_MSM_SHORT_BELOW;
    return len < below ? 0 : msm_window_bits(group, len);
}

struct MsmPlan {
    std::vector<MsmSeg> segs;
    std::vector<uint32_t> idx;  // the Straus segments, then the Pippenger ones
    std::vector<MsmWin> wins;
    size_t nstraus = 0, entries = 0, nbuckets = 0, straus_terms = 0;
    int key_bits = 1;
};

// offsets already checked (msm_offsets_args).  force_c < 0: every segment as msm_segment_c plans it; otherwise every non-empty segment
// on the path force_c names (0 Straus, else Pippenger with force_c-bit windows: sipp_test_msm_batch_device, which times both paths)
int msm_plan(int group, const size_t* offsets, size_t count, MsmPlan& p, int force_c = -1) {
    const GroupInfo g = group_info(group);
    const size_t n = offsets[count];
    if (count > (size_t)UINT32_MAX) return fail(SIPP_ERR_CUDA, "msm_batch: more than 2^32 - 1 segments are not supported");
    if (n * g.nc >= ((size_t)1 << 31)) return fail(SIPP_ERR_CUDA, "msm_batch: the device scratch of more than 2^31 terms is not supported");
    p.segs.resize(count);
    std::vector<uint32_t> pipp;
    size_t parts_total = 0;
    for (size_t j = 0; j < count; j++) {
        const size_t len = offsets[j + 1] - offsets[j];
        MsmSeg& s = p.segs[j];
        const int c = force_c < 0 || len == 0 ? msm_segment_c(group, len) : force_c;
        s = MsmSeg{(uint32_t)offsets[j], (uint32_t)len, (uint32_t)c, 0, 0, 0, 0, 0};
        if (s.c == 0) {
            p.idx.push_back((uint32_t)j);
            p.straus_terms += len * g.nc;
            continue;
        }
        pipp.push_back((uint32_t)j);
        const size_t W = (size_t)windows_of(g, (int)s.c), nb = buckets_of(g, (int)s.c);
        const size_t span = (size_t)64 * SIPP_MSM_BUCKETS_PER_THREAD;
        s.parts = (uint32_t)((nb + span - 1) / span);
        s.ebase = (uint32_t)p.entries;
        s.bbase = (uint32_t)p.nbuckets;
        s.wbase = (uint32_t)parts_total;
        for (size_t w = 0; w < W; w++)
            for (uint32_t q = 0; q < s.parts; q++) {
                const size_t lo = q * span, cnt = nb - lo < span ? nb - lo : span;
                p.wins.push_back(MsmWin{(uint32_t)(p.nbuckets + w * nb), (uint32_t)lo, (uint32_t)cnt, 0});
            }
        p.entries += len * g.nc * W;
        p.nbuckets += W * nb;
        parts_total += W * s.parts;
        if (p.entries >= ((size_t)1 << 31) || p.nbuckets >= ((size_t)1 << 31))
            return fail(SIPP_ERR_CUDA, "msm_batch: the device scratch of more than 2^31 sort entries or buckets is not supported");
    }
    p.nstraus = p.idx.size();
    p.idx.insert(p.idx.end(), pipp.begin(), pipp.end());
    while (((size_t)1 << p.key_bits) <= p.nbuckets) p.key_bits++;  // keys 0 .. nbuckets (the zero-digit key) sort on key_bits bits
    return SIPP_OK;
}

// the offsets rules of sipp_inner_product_batch, then the 2^32 - 1 point limit (count > 0, offsets not NULL)
int msm_offsets_args(size_t n, const size_t* offsets, size_t count) {
    if (offsets[0] != 0) return fail(SIPP_ERR_ARG, "msm_batch: offsets[0] != 0");
    for (size_t j = 0; j < count; j++)
        if (offsets[j + 1] < offsets[j]) return fail(SIPP_ERR_ARG, "msm_batch: decreasing offsets");
    if (offsets[count] != n) return fail(SIPP_ERR_ARG, "msm_batch: offsets[count] != number of points");
    if (n > (size_t)UINT32_MAX) return fail(SIPP_ERR_ARG, "msm_batch: more than 2^32 - 1 points");
    return SIPP_OK;
}

int msm_args(const void* points, const void* scalars, size_t n, const size_t* offsets, size_t count, const void* out) {
    if (count == 0) return n == 0 ? SIPP_OK : fail(SIPP_ERR_ARG, "msm_batch: count == 0 with points");
    if (!points || !scalars || !offsets || !out) return fail(SIPP_ERR_ARG, "msm_batch: null pointer");
    return msm_offsets_args(n, offsets, count);
}

bool scalars_canonical(const uint8_t* k, size_t count) {  // every 32-byte little-endian scalar < r
    static const uint64_t RM[4] = {0x43e1f593f0000001ull, 0x2833e84879b97091ull, 0xb85045b68181585dull, 0x30644e72e131a029ull};
    for (size_t i = 0; i < count; i++) {
        uint64_t w[4];
        memcpy(w, k + 32 * i, 32);
        bool less = false;
        for (int j = 3; j >= 0; j--) {
            if (w[j] != RM[j]) { less = w[j] < RM[j]; break; }
        }
        if (!less) return false;
    }
    return true;
}

// the whole call on the device: points / scalars hold the boundary bytes (the caller's buffers or staging copies); the results
// (boundary bytes) are copied to `out` (host or device memory, per out_kind) only when every input passed its checks
int msm_run(int group, const uint32_t* points, const uint32_t* scalars, size_t n, const size_t* offsets, size_t count, void* out,
            cudaMemcpyKind out_kind, int force_c = -1) {
    cudaStream_t s = g_stream;
    const GroupInfo g = group_info(group);
    MsmPlan plan;
    int rc = msm_plan(group, offsets, count, plan, force_c);
    if (rc) return rc;
    const size_t nterms = n * g.nc, entries = plan.entries;
    size_t sort_bytes = 0;
    if (entries) {
        const int le = msm_sort(nullptr, &sort_bytes, nullptr, nullptr, nullptr, nullptr, (uint32_t)entries, plan.key_bits, s);
        if (le) return cuda_fail((cudaError_t)le, "msm_batch: sort scratch");
    }
    std::vector<void*> blocks;
    struct Release {
        std::vector<void*>& p;
        ~Release() { for (void* q : p) pool_free(q); }  // recycled blocks: later work on the same stream only
    } release{blocks};
    cudaError_t e = cudaSuccess;
    auto get = [&](void** ptr, size_t bytes) {
        *ptr = nullptr;
        if (e == cudaSuccess && bytes) {
            e = pool_alloc(ptr, bytes);
            if (e == cudaSuccess) blocks.push_back(*ptr);
        }
    };
    uint32_t *mp, *mo, *enc, *keys, *vals, *keys2, *vals2, *idx;
    void *terms, *buckets, *parts, *temp;
    FoldComp* naf;
    MsmSeg* dsegs;
    MsmWin* dwins;
    int* flags;
    get((void**)&mp, n * g.words * 4);
    get(&terms, nterms * msm_term_bytes(group));
    get((void**)&naf, plan.straus_terms ? nterms * sizeof(FoldComp) : 0);
    get((void**)&keys, entries * 4);
    get((void**)&vals, entries * 4);
    get((void**)&keys2, entries * 4);
    get((void**)&vals2, entries * 4);
    get(&temp, sort_bytes);
    get(&buckets, plan.nbuckets * msm_jac_bytes(group));
    void *first, *last;
    const size_t chunks = (entries + SIPP_MSM_CHUNK - 1) / SIPP_MSM_CHUNK;
    get(&first, chunks * msm_jac_bytes(group));
    get(&last, chunks * msm_jac_bytes(group));
    uint32_t* long_list;
    void* long_parts;
    get((void**)&long_list, entries ? msm_long_list_words((uint32_t)entries) * 4 : 0);
    get(&long_parts, entries ? (msm_long_list_words((uint32_t)entries) - 1) * SIPP_MSM_LONG_PARTS * msm_jac_bytes(group) : 0);
    get(&parts, plan.wins.size() * msm_jac_bytes(group));
    get((void**)&mo, count * g.words * 4);
    get((void**)&enc, count * g.words * 4);
    get((void**)&dsegs, count * sizeof(MsmSeg));
    get((void**)&dwins, plan.wins.size() * sizeof(MsmWin));
    get((void**)&idx, count * sizeof(uint32_t));
    get((void**)&flags, sizeof(int));
    if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(msm_batch)");
    auto run = [&]() -> int {
        CK(cudaMemsetAsync(flags, 0, sizeof(int), s));
        CK(cudaMemcpyAsync(dsegs, plan.segs.data(), count * sizeof(MsmSeg), cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(idx, plan.idx.data(), count * sizeof(uint32_t), cudaMemcpyHostToDevice, s));
        if (!plan.wins.empty()) CK(cudaMemcpyAsync(dwins, plan.wins.data(), plan.wins.size() * sizeof(MsmWin), cudaMemcpyHostToDevice, s));
        const int words = g.words;
        int le = 0;
        if (n) {
            le = launch_codec_decode(points, mp, n * (words / 8), flags, s);
            if (!le && g_opt_validate)  // on the curve, G2 points in the order-r subgroup (SIPP_OPT_VALIDATE_POINTS), as sipp_inner_product
                le = launch_validate_points_groups(group == 1 ? mp : nullptr, group == 1 ? n : 0, group == 2 ? mp : nullptr, group == 2 ? n : 0, flags, s);
            if (!le) le = launch_msm_recode(group, mp, scalars, (uint32_t)n, dsegs, (uint32_t)count, terms, naf, keys, vals, (uint32_t)plan.nbuckets, flags, s);
            if (le) return cuda_fail((cudaError_t)le, "k_msm_recode");
            g_stats.launches += g_opt_validate ? 3 : 2;
        }
        if (entries) {
            le = msm_sort(temp, &sort_bytes, keys, keys2, vals, vals2, (uint32_t)entries, plan.key_bits, s);
            if (le) return cuda_fail((cudaError_t)le, "msm_batch: sort");
            CK(cudaMemsetAsync(buckets, 0, plan.nbuckets * msm_jac_bytes(group), s));  // all-zero words: z = 0, the identity
            le = launch_msm_buckets(group, keys2, vals2, (uint32_t)entries, (uint32_t)plan.nbuckets, terms, buckets, first, last, long_list, long_parts, s);
            if (!le) le = launch_msm_windows(group, buckets, dwins, (uint32_t)plan.wins.size(), parts, s);
            if (!le) le = launch_msm_finish(group, parts, dsegs, idx + plan.nstraus, (uint32_t)(count - plan.nstraus), mo, s);
            if (le) return cuda_fail((cudaError_t)le, "k_msm_buckets / k_msm_windows / k_msm_finish");
            g_stats.launches += 7;
        }
        if (plan.nstraus) {
            le = launch_msm_straus(group, terms, naf, dsegs, idx, (uint32_t)plan.nstraus, mo, s);
            if (le) return cuda_fail((cudaError_t)le, "k_msm_straus");
            g_stats.launches++;
        }
        int flag = 0;
        CK(cudaMemcpyAsync(&flag, flags, sizeof(int), cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        // the precedence of the host forms: a scalar >= r first, then a coordinate >= p, then the point checks
        if (flag & 8) return fail(SIPP_ERR_ENCODING, "scalar >= r");
        if (flag & 16) return fail(SIPP_ERR_ENCODING, "scalar decomposition out of range (not expected for any scalar < r)");
        if (flag & 1) return fail(SIPP_ERR_ENCODING, "input coordinate >= p");
        if (flag & 2) return fail(SIPP_ERR_ENCODING, "input point is not on the curve");
        if (flag & 4) return fail(SIPP_ERR_ENCODING, "input G2 point is not in the prime-order subgroup");
        le = launch_codec_encode(mo, enc, count * (words / 8), s);
        if (le) return cuda_fail((cudaError_t)le, "k_codec_encode");
        g_stats.launches++;
        CK(cudaMemcpyAsync(out, enc, count * words * 4, out_kind, s));
        CK(cudaStreamSynchronize(s));
        return SIPP_OK;
    };
    rc = run();
    if (rc) cudaStreamSynchronize(s);
    return rc;
}

int msm_host(int group, const uint8_t* points, const uint8_t* scalars, size_t n, const size_t* offsets, size_t count, uint8_t* out) {
    int rc = msm_args(points, scalars, n, offsets, count, out);
    if (rc || count == 0) return rc ? rc : ensure_init();
    const size_t pbytes = group == 1 ? 64 : 128;
    if (!scalars_canonical(scalars, n)) return fail(SIPP_ERR_ENCODING, "scalar >= r");
    if (!fq_bytes_canonical(points, n * (pbytes / 32))) return fail(SIPP_ERR_ENCODING, "input coordinate >= p");
    rc = ensure_init();
    if (rc) return rc;
    uint8_t *tp = nullptr, *tk = nullptr;
    cudaError_t e = pool_alloc((void**)&tp, n ? n * pbytes : 1);
    if (e == cudaSuccess) e = pool_alloc((void**)&tk, n ? n * 32 : 1);
    struct Release {
        uint8_t *a, *b;
        ~Release() { pool_free(a); pool_free(b); }
    } release{tp, tk};
    if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(msm_batch)");
    if (n) {
        CK(cudaMemcpyAsync(tp, points, n * pbytes, cudaMemcpyHostToDevice, g_stream));
        CK(cudaMemcpyAsync(tk, scalars, n * 32, cudaMemcpyHostToDevice, g_stream));
    }
    return msm_run(group, (const uint32_t*)tp, (const uint32_t*)tk, n, offsets, count, out, cudaMemcpyDeviceToHost);  // synchronises
}

int msm_device(int group, const void* d_points, const void* d_scalars, size_t n, const size_t* offsets, size_t count, void* d_out,
               int force_c = -1) {
    int rc = msm_args(d_points, d_scalars, n, offsets, count, d_out);
    if (rc || count == 0) return rc ? rc : ensure_init();
    rc = ensure_init();
    if (rc) return rc;
    CK(order_after(g_stream, cudaStreamLegacy));  // inputs just written on the legacy default stream (torch's, unless switched)
    return msm_run(group, (const uint32_t*)d_points, (const uint32_t*)d_scalars, n, offsets, count, d_out, cudaMemcpyDeviceToDevice, force_c);
}

// the GT multi-exponentiation on the device: elems / scalars hold the boundary bytes (the caller's buffers or staging copies); the
// results (boundary bytes) are copied to `out` (host or device memory, per out_kind) only when every input passed its checks
int gt_msm_run(const uint32_t* elems, const uint32_t* scalars, size_t n, const size_t* offsets, size_t count, void* out, cudaMemcpyKind out_kind,
               int force_c = -1) {
    cudaStream_t s = g_stream;
    MsmPlan plan;
    int rc = msm_plan(3, offsets, count, plan, force_c);
    if (rc) return rc;
    // the segmented product over the table slots: a short-path segment multiplies its powered elements, a Pippenger segment its one
    // result (k_gt_msm_finish writes it to the slot of its first element), an empty segment gives 1
    std::vector<size_t> start(count), len(count);
    std::vector<uint32_t> pow_idx;
    pow_idx.reserve(plan.straus_terms);
    for (size_t j = 0; j < count; j++) {
        const MsmSeg& sg = plan.segs[j];
        start[j] = sg.first;
        len[j] = sg.c ? 1 : sg.len;
        if (sg.c == 0)
            for (uint32_t i = 0; i < sg.len; i++) pow_idx.push_back(sg.first + i);
    }
    std::vector<ProductTask> tasks;
    std::vector<size_t> pass_first;
    const size_t seg0 = seg_product_tasks(start, len, n, tasks, pass_first);
    const size_t entries = plan.entries, npipp = count - plan.nstraus, fq12 = 384;
    size_t sort_bytes = 0;
    if (entries) {
        const int le = msm_sort(nullptr, &sort_bytes, nullptr, nullptr, nullptr, nullptr, (uint32_t)entries, plan.key_bits, s);
        if (le) return cuda_fail((cudaError_t)le, "gt_msm_batch: sort scratch");
    }
    std::vector<void*> blocks;
    struct Release {
        std::vector<void*>& p;
        ~Release() { for (void* q : p) pool_free(q); }  // recycled blocks: later work on the same stream only
    } release{blocks};
    cudaError_t e = cudaSuccess;
    auto get = [&](void** ptr, size_t bytes) {
        *ptr = nullptr;
        if (e == cudaSuccess && bytes) {
            e = pool_alloc(ptr, bytes);
            if (e == cudaSuccess) blocks.push_back(*ptr);
        }
    };
    const size_t chunks = (entries + SIPP_MSM_CHUNK - 1) / SIPP_MSM_CHUNK, lwords = entries ? msm_long_list_words((uint32_t)entries) : 0;
    uint32_t *table, *sc, *keys, *vals, *keys2, *vals2, *buckets, *first, *last, *long_list, *long_parts, *parts, *enc, *idx, *dpow;
    void* temp;
    MsmSeg* dsegs;
    MsmWin* dwins;
    ProductTask* dtasks;
    int* flags;
    get((void**)&table, (seg0 + count) * fq12);
    get((void**)&sc, pow_idx.size() ? n * 32 : 0);
    get((void**)&keys, entries * 4);
    get((void**)&vals, entries * 4);
    get((void**)&keys2, entries * 4);
    get((void**)&vals2, entries * 4);
    get(&temp, sort_bytes);
    get((void**)&buckets, plan.nbuckets * fq12);
    get((void**)&first, chunks * fq12);
    get((void**)&last, chunks * fq12);
    get((void**)&long_list, lwords * 4);
    get((void**)&long_parts, lwords ? (lwords - 1) * SIPP_MSM_LONG_PARTS * fq12 : 0);
    get((void**)&parts, plan.wins.size() * fq12);
    get((void**)&enc, count * fq12);
    get((void**)&dsegs, count * sizeof(MsmSeg));
    get((void**)&dwins, plan.wins.size() * sizeof(MsmWin));
    get((void**)&idx, count * sizeof(uint32_t));
    get((void**)&dpow, pow_idx.size() * sizeof(uint32_t));
    get((void**)&dtasks, tasks.size() * sizeof(ProductTask));
    get((void**)&flags, sizeof(int));
    if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(gt_msm_batch)");
    auto run = [&]() -> int {
        CK(cudaMemsetAsync(flags, 0, sizeof(int), s));
        CK(cudaMemcpyAsync(dsegs, plan.segs.data(), count * sizeof(MsmSeg), cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(idx, plan.idx.data(), count * sizeof(uint32_t), cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(dtasks, tasks.data(), tasks.size() * sizeof(ProductTask), cudaMemcpyHostToDevice, s));
        if (!plan.wins.empty()) CK(cudaMemcpyAsync(dwins, plan.wins.data(), plan.wins.size() * sizeof(MsmWin), cudaMemcpyHostToDevice, s));
        if (!pow_idx.empty()) CK(cudaMemcpyAsync(dpow, pow_idx.data(), pow_idx.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, s));
        int le = 0;
        if (n) {
            le = launch_gt_msm_decode(elems, scalars, (uint32_t)n, dsegs, (uint32_t)count, table, sc, keys, vals, (uint32_t)plan.nbuckets, flags, s);
            if (le) return cuda_fail((cudaError_t)le, "k_gt_msm_decode");
            g_stats.launches++;
        }
        if (entries) {
            le = msm_sort(temp, &sort_bytes, keys, keys2, vals, vals2, (uint32_t)entries, plan.key_bits, s);
            if (le) return cuda_fail((cudaError_t)le, "gt_msm_batch: sort");
            le = launch_gt_msm_buckets(keys2, vals2, (uint32_t)entries, (uint32_t)plan.nbuckets, table, buckets, first, last, long_list, long_parts, s);
            if (!le) le = launch_gt_msm_windows(buckets, dwins, (uint32_t)plan.wins.size(), parts, (uint32_t)npipp, dsegs, idx + plan.nstraus, table, s);
            if (le) return cuda_fail((cudaError_t)le, "k_gt_msm_buckets / k_gt_msm_windows / k_gt_msm_finish");
            g_stats.launches += 8;
        }
        if (!pow_idx.empty()) {
            le = launch_gt_msm_pow(table, (const uint64_t*)sc, dpow, pow_idx.size(), s);
            if (le) return cuda_fail((cudaError_t)le, "k_gt_msm_pow");
            g_stats.launches++;
        }
        for (size_t k = 0; k + 1 < pass_first.size(); k++) {
            le = launch_seg_product(dtasks + pass_first[k], pass_first[k + 1] - pass_first[k], table, s);
            if (le) return cuda_fail((cudaError_t)le, "k_seg_product");
            g_stats.launches++;
        }
        int flag = 0;
        CK(cudaMemcpyAsync(&flag, flags, sizeof(int), cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        // the precedence of the host forms: a scalar >= r first, then a coordinate >= p
        if (flag & 8) return fail(SIPP_ERR_ENCODING, "scalar >= r");
        if (flag & 1) return fail(SIPP_ERR_ENCODING, "input coordinate >= p");
        le = launch_gt_msm_encode(table + seg0 * 96, count, enc, s);
        if (le) return cuda_fail((cudaError_t)le, "k_gt_msm_encode");
        g_stats.launches++;
        CK(cudaMemcpyAsync(out, enc, count * fq12, out_kind, s));
        CK(cudaStreamSynchronize(s));
        return SIPP_OK;
    };
    rc = run();
    if (rc) cudaStreamSynchronize(s);
    return rc;
}

int gt_msm_host(const uint8_t* elems, const uint8_t* scalars, size_t n, const size_t* offsets, size_t count, uint8_t* out) {
    int rc = msm_args(elems, scalars, n, offsets, count, out);
    if (rc || count == 0) return rc ? rc : ensure_init();
    if (!scalars_canonical(scalars, n)) return fail(SIPP_ERR_ENCODING, "scalar >= r");
    if (!fq_bytes_canonical(elems, n * 12)) return fail(SIPP_ERR_ENCODING, "input coordinate >= p");
    rc = ensure_init();
    if (rc) return rc;
    uint8_t *te = nullptr, *tk = nullptr;
    cudaError_t e = pool_alloc((void**)&te, n ? n * 384 : 1);
    if (e == cudaSuccess) e = pool_alloc((void**)&tk, n ? n * 32 : 1);
    struct Release {
        uint8_t *a, *b;
        ~Release() { pool_free(a); pool_free(b); }
    } release{te, tk};
    if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(gt_msm_batch)");
    if (n) {
        CK(cudaMemcpyAsync(te, elems, n * 384, cudaMemcpyHostToDevice, g_stream));
        CK(cudaMemcpyAsync(tk, scalars, n * 32, cudaMemcpyHostToDevice, g_stream));
    }
    return gt_msm_run((const uint32_t*)te, (const uint32_t*)tk, n, offsets, count, out, cudaMemcpyDeviceToHost);  // synchronises
}

int gt_msm_device(const void* d_elems, const void* d_scalars, size_t n, const size_t* offsets, size_t count, void* d_out, int force_c = -1) {
    int rc = msm_args(d_elems, d_scalars, n, offsets, count, d_out);
    if (rc || count == 0) return rc ? rc : ensure_init();
    rc = ensure_init();
    if (rc) return rc;
    CK(order_after(g_stream, cudaStreamLegacy));  // inputs just written on the legacy default stream (torch's, unless switched)
    return gt_msm_run((const uint32_t*)d_elems, (const uint32_t*)d_scalars, n, offsets, count, d_out, cudaMemcpyDeviceToDevice, force_c);
}

}  // namespace

extern "C" {

int sipp_g1_msm_batch(const uint8_t* points, const uint8_t* scalars, size_t n, const size_t* offsets, size_t count, uint8_t* out) {
    return msm_host(1, points, scalars, n, offsets, count, out);
}
int sipp_g2_msm_batch(const uint8_t* points, const uint8_t* scalars, size_t n, const size_t* offsets, size_t count, uint8_t* out) {
    return msm_host(2, points, scalars, n, offsets, count, out);
}
int sipp_g1_msm_batch_device(const void* d_points, const void* d_scalars, size_t n, const size_t* offsets, size_t count, void* d_out) {
    return msm_device(1, d_points, d_scalars, n, offsets, count, d_out);
}
int sipp_g2_msm_batch_device(const void* d_points, const void* d_scalars, size_t n, const size_t* offsets, size_t count, void* d_out) {
    return msm_device(2, d_points, d_scalars, n, offsets, count, d_out);
}

// host-only plan of a batch (no GPU needed): 4 words per segment -- G1 path (0 Straus, 1 Pippenger), G1 window bits (0 for Straus), then
// the same for G2 -- to `out` when out_cap >= 4 x count; returns count or a negative status (the offsets checks of the entry points)
long sipp_test_msm_plan(const size_t* offsets, size_t count, int* out, size_t out_cap) {
    if (!offsets) return fail(SIPP_ERR_ARG, "null offsets");
    if (count == 0) return 0;
    const size_t n = offsets[count];
    int rc = msm_offsets_args(n, offsets, count);
    if (rc) return rc;
    if (out && out_cap >= 4 * count) {
        for (size_t j = 0; j < count; j++) {
            const size_t len = offsets[j + 1] - offsets[j];
            for (int group = 1; group <= 2; group++) {
                const int c = msm_segment_c(group, len);
                out[4 * j + 2 * (group - 1)] = c ? 1 : 0;
                out[4 * j + 2 * (group - 1) + 1] = c;
            }
        }
    }
    return (long)count;
}

// the device form with every non-empty segment forced onto one path: c = 0 Straus, SIPP_MSM_MIN_C <= c <= SIPP_MSM_MAX_C Pippenger with
// c-bit windows (any other c: SIPP_ERR_ARG, after the checks of the device form).  Same outputs as the plan's path; for timing the
// two paths at the same segment length.
int sipp_test_msm_batch_device(int group, int c, const void* d_points, const void* d_scalars, size_t n, const size_t* offsets, size_t count,
                               void* d_out) {
    if (group != 1 && group != 2) return fail(SIPP_ERR_ARG, "group must be 1 or 2");
    if (c != 0 && (c < SIPP_MSM_MIN_C || c > SIPP_MSM_MAX_C)) return fail(SIPP_ERR_ARG, "c must be 0 or 5 .. 16");
    return msm_device(group, d_points, d_scalars, n, offsets, count, d_out, c);
}

int sipp_gt_msm_batch(const uint8_t* elems, const uint8_t* scalars, size_t n, const size_t* offsets, size_t count, uint8_t* out) {
    return gt_msm_host(elems, scalars, n, offsets, count, out);
}
int sipp_gt_msm_batch_device(const void* d_elems, const void* d_scalars, size_t n, const size_t* offsets, size_t count, void* d_out) {
    return gt_msm_device(d_elems, d_scalars, n, offsets, count, d_out);
}

// host-only plan of a GT batch (no GPU needed): 2 words per segment -- path (0 short, 1 Pippenger), window bits (0 for the short path) --
// to `out` when out_cap >= 2 x count; returns count or a negative status (the offsets checks of the entry points)
long sipp_test_gt_msm_plan(const size_t* offsets, size_t count, int* out, size_t out_cap) {
    if (!offsets) return fail(SIPP_ERR_ARG, "null offsets");
    if (count == 0) return 0;
    int rc = msm_offsets_args(offsets[count], offsets, count);
    if (rc) return rc;
    if (out && out_cap >= 2 * count) {
        for (size_t j = 0; j < count; j++) {
            const int c = msm_segment_c(3, offsets[j + 1] - offsets[j]);
            out[2 * j] = c ? 1 : 0;
            out[2 * j + 1] = c;
        }
    }
    return (long)count;
}

// sipp_gt_msm_batch_device with every non-empty segment forced onto one path: c = 0 the short path, SIPP_GT_MSM_MIN_C <= c <=
// SIPP_MSM_MAX_C Pippenger with c-bit windows (any other c: SIPP_ERR_ARG, before the checks of the device form).  Same outputs as the
// plan's path; for timing both paths at the same segment length.
int sipp_test_gt_msm_batch_device(int c, const void* d_elems, const void* d_scalars, size_t n, const size_t* offsets, size_t count, void* d_out) {
    if (c != 0 && (c < SIPP_GT_MSM_MIN_C || c > SIPP_MSM_MAX_C)) return fail(SIPP_ERR_ARG, "c must be 0 or 2 .. 16");
    return gt_msm_device(d_elems, d_scalars, n, offsets, count, d_out, c);
}

}  // extern "C"

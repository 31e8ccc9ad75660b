// ragged.cu -- batched proving and verification of independent instances of different sizes (C ABI: sipp_prove_native_batch_ragged,
// sipp_prove_native_batch_ragged_device, their _statement forms, sipp_verify_native_batch_ragged, test hook sipp_test_ragged_schedule).
//
// Instance j is pairs [offsets[j], offsets[j + 1]) of A and B, n_j a power of two; its proof is exactly sipp_prove_native on those
// pairs (prover_native.rs:26-80).  The instances run in lock-step rounds, as in batch.cu, but each with its own size:
//   order       the instances sorted by n descending (stable): the instances of round r >= 1 (log2 n_j >= r) are a prefix of it.
//               An index permutation only -- no point moves, every proof lands in the caller's order.
//   schedule    every round's product plan, fold table and proof-slot table is built on the host before the first launch and
//               uploaded once; nothing returns to the host until the final flag check.
//   round 0     Z of every instance: the products path (products.h) directly on the decoded points, whose segments are the instances.
//   round r     k_ragged_gather writes A_hi || A_lo, B_lo || B_hi of every active instance (current size m = n_j >> (r - 1), h = m / 2)
//               to scratch, so Z_L = <A_hi, B_lo> and Z_R = <A_lo, B_hi> are two consecutive segments of the same products path;
//               k_scatter_fq12 puts the products in their proof slots, k_tr_round_ragged absorbs them and recodes the challenge,
//               and a ragged fold kernel (k_fold_*_ragged, chosen by the round's element count as in batch.cu) folds in place.
// The registration of A and B (k_tr_absorb_pairs_ragged) is 8 n_j strictly serial permutations per instance, so the LONGEST instance
// bounds it: an instance far larger than the rest is better proved on its own with sipp_prove_native, whose chain runs on the host.
// The verifier (ragged_verify_run) shares the order, the fold tables and kernels, the absorb and the transcript round.
#include <string.h>

#include <algorithm>
#include <vector>

#include "products.h"

using namespace sipp;
using namespace sipp_host;

namespace {

struct RaggedRound {
    size_t act = 0;               // instances of the round: positions [0, act) of the order
    size_t pairs = 0;             // pairs of its products
    size_t elems = 0, units = 0;  // fold elements and wide-fold units (rounds >= 1)
    int kernel = -1;              // fold kernel: -1 none, 0 k_fold_batch, 1 k_fold_wide_batch, 2 k_fold_straus (ragged forms)
    size_t tab0 = 0, dst0 = 0;    // first entries of its fold table and of its proof-slot destinations
    size_t g0 = 0, t0 = 0;        // first entries of its groups and tasks in the uploaded arrays
    ProductPlan plan;
};

struct RaggedSchedule {
    std::vector<size_t> order;        // instance index at each position, n descending (stable)
    std::vector<RaggedProof> proofs;  // by position
    size_t proof_fq12 = 0;            // sum of np_j
    std::vector<RaggedInst> tabs;     // fold tables of rounds >= 1, concatenated
    std::vector<uint64_t> dst;        // proof slot of every product of every round, concatenated
    std::vector<ProductGroup> groups;
    std::vector<ProductTask> tasks;
    std::vector<RaggedRound> rounds;  // 0 .. log2 max n_j
    size_t lines_pairs = 0, work_slots = 0, max_products = 0;
};

size_t log2_of(size_t v) {
    size_t r = 0;
    while (((size_t)1 << r) < v) r++;
    return r;
}

int ragged_args(const void* A, size_t a_len, const void* B, size_t b_len, const size_t* offsets, size_t count, const void* proofs) {
    if (a_len != b_len) return fail(SIPP_ERR_LENGTH, "assert_eq!(A.len(), B.len())");
    if (!A || !B || !offsets || !proofs || count == 0) return fail(SIPP_ERR_ARG, "prove_native_batch_ragged: null pointer or count == 0");
    if (offsets[0] != 0) return fail(SIPP_ERR_ARG, "prove_native_batch_ragged: offsets[0] != 0");
    for (size_t j = 0; j < count; j++)
        if (offsets[j + 1] < offsets[j]) return fail(SIPP_ERR_ARG, "prove_native_batch_ragged: decreasing offsets");
    if (offsets[count] != a_len) return fail(SIPP_ERR_ARG, "prove_native_batch_ragged: offsets[count] != number of pairs");
    for (size_t j = 0; j < count; j++)
        if (!is_pow2(offsets[j + 1] - offsets[j])) return fail(SIPP_ERR_ARG, "prove_native_batch_ragged: n_j must be a non-zero power of two");
    if (a_len > (size_t)UINT32_MAX) return fail(SIPP_ERR_ARG, "prove_native_batch_ragged: more than 2^32 - 1 pairs");
    return SIPP_OK;
}

// the fold side of the schedule, which the verifier shares: the order, every round's active instances, fold elements, wide-fold
// units and fold kernel, and the fold tables of rounds >= 1.  offsets already checked (ragged_args); reads the fold thresholds
void ragged_folds(const size_t* offsets, size_t count, RaggedSchedule& S) {
    std::vector<size_t> n(count);
    for (size_t j = 0; j < count; j++) n[j] = offsets[j + 1] - offsets[j];
    S.order.resize(count);
    for (size_t j = 0; j < count; j++) S.order[j] = j;
    std::stable_sort(S.order.begin(), S.order.end(), [&](size_t a, size_t b) { return n[a] > n[b]; });
    const size_t R = log2_of(n[S.order[0]]);
    S.rounds.assign(R + 1, RaggedRound());
    S.tabs.clear();
    S.rounds[0].act = count;
    size_t act = count;
    for (size_t r = 1; r <= R; r++) {
        RaggedRound& rd = S.rounds[r];
        while (act > 0 && n[S.order[act - 1]] < ((size_t)1 << r)) act--;
        rd.act = act;
        rd.tab0 = S.tabs.size();
        for (size_t k = 0; k < act; k++) {
            const size_t j = S.order[k], h = n[j] >> r;
            S.tabs.push_back(RaggedInst{(uint32_t)rd.elems, (uint32_t)rd.units, (uint32_t)h, (uint32_t)offsets[j]});
            rd.elems += h;
            rd.units += (h & 1) ? 1 : h / 2;
        }
        // the thresholds of batch.cu: one thread per element when the launch fills the GPU, the lane engine up to two waves
        rd.kernel = (g_opt_fold_straus && rd.elems >= 16384) ? 2 : rd.elems <= (size_t)g_opt_wide_fold_max + 512 ? 1 : 0;
    }
}

// the prover's schedule: the fold side (ragged_folds), the proof slots and every round's product plan.  offsets already checked
// (ragged_args); reads the options of the products path and the fold thresholds
int ragged_schedule(const size_t* offsets, size_t count, RaggedSchedule& S) {
    ragged_folds(offsets, count, S);
    std::vector<size_t> n(count), first(count);
    for (size_t j = 0; j < count; j++) n[j] = offsets[j + 1] - offsets[j];
    S.proof_fq12 = 0;
    for (size_t j = 0; j < count; j++) {
        first[j] = S.proof_fq12;
        S.proof_fq12 += sipp_proof_len(n[j]);
    }
    S.proofs.resize(count);
    for (size_t k = 0; k < count; k++) S.proofs[k] = RaggedProof{first[S.order[k]], (uint32_t)sipp_proof_len(n[S.order[k]]), 0};
    const size_t R = S.rounds.size() - 1;
    S.dst.clear(); S.groups.clear(); S.tasks.clear();
    S.lines_pairs = S.work_slots = S.max_products = 0;
    auto add_plan = [&](RaggedRound& rd, const size_t* offs, size_t nprod) -> int {
        int rc = product_plan(offs, nprod, g_opt_batch_kpg_max, (size_t)g_opt_product_chunk, rd.plan);
        if (rc) return rc;
        rd.g0 = S.groups.size();
        rd.t0 = S.tasks.size();
        S.groups.insert(S.groups.end(), rd.plan.groups.begin(), rd.plan.groups.end());
        S.tasks.insert(S.tasks.end(), rd.plan.tasks.begin(), rd.plan.tasks.end());
        const size_t lp = rd.pairs < rd.plan.chunk_pairs ? rd.pairs : rd.plan.chunk_pairs;
        S.lines_pairs = std::max(S.lines_pairs, lp);
        S.work_slots = std::max(S.work_slots, rd.plan.work_slots(nprod));
        S.max_products = std::max(S.max_products, nprod);
        return SIPP_OK;
    };
    // round 0: Z of every instance (slot np_j - 1), the caller's segments as they are
    RaggedRound& r0 = S.rounds[0];
    r0.pairs = offsets[count];
    r0.dst0 = 0;
    for (size_t j = 0; j < count; j++) S.dst.push_back(first[j] + sipp_proof_len(n[j]) - 1);
    int rc = add_plan(r0, offsets, count);
    if (rc) return rc;
    std::vector<size_t> offs;
    for (size_t r = 1; r <= R; r++) {
        RaggedRound& rd = S.rounds[r];
        rd.dst0 = S.dst.size();
        offs.assign(1, 0);
        for (size_t k = 0; k < rd.act; k++) {
            const size_t j = S.order[k], h = n[j] >> r;
            offs.push_back(offs.back() + h);  // Z_L = <A_hi, B_lo>
            offs.push_back(offs.back() + h);  // Z_R = <A_lo, B_hi>
            const size_t np = sipp_proof_len(n[j]);
            S.dst.push_back(first[j] + np - 2 * r);      // proof.reverse()  prover_native.rs:78
            S.dst.push_back(first[j] + np - 1 - 2 * r);
        }
        rd.pairs = 2 * rd.elems;
        rc = add_plan(rd, offs.data(), 2 * rd.act);
        if (rc) return rc;
    }
    return SIPP_OK;
}

// decode (and, with SIPP_OPT_VALIDATE_POINTS, check) the n points of both sides into dA / dB, flags[1] recording a bad point, and
// register A and B (prover_native.rs:36-39, verifier_native.rs:25-28) of the act1 instances with n_j >= 2 (round 1's table tab1)
int ragged_decode_absorb(const uint32_t* bytesA, const uint32_t* bytesB, size_t n, uint32_t* dA, uint32_t* dB, const RaggedInst* tab1, size_t act1,
                         uint64_t* states, int* flags, cudaStream_t s) {
    Span sp(3, s);
    int le = launch_codec_decode(bytesA, dA, n * 2, flags + 1, s);
    if (!le) le = launch_codec_decode(bytesB, dB, n * 4, flags + 1, s);
    if (le) return cuda_fail((cudaError_t)le, "k_codec_decode");
    g_stats.launches += 2;
    if (g_opt_validate) {  // on the curve, B_i in the order-r subgroup (SIPP_OPT_VALIDATE_POINTS)
        le = launch_validate_points(dA, dB, n, flags + 1, s);
        if (le) return cuda_fail((cudaError_t)le, "k_validate_points");
        g_stats.launches++;
    }
    if (act1) {
        le = launch_tr_absorb_pairs_ragged(bytesA, bytesB, tab1, (unsigned)act1, states, s);
        if (le) return cuda_fail((cudaError_t)le, "k_tr_absorb_pairs_ragged");
        g_stats.launches++;
    }
    return SIPP_OK;
}

// the status of a finished call from its flags: [0] transcript / recoding, [1] encoding
int ragged_flags_status(const int fl[2]) {
    if (fl[1] & 1) return fail(SIPP_ERR_ENCODING, "input coordinate >= p");
    if (fl[1] & 2) return fail(SIPP_ERR_ENCODING, "input point is not on the curve");
    if (fl[1] & 4) return fail(SIPP_ERR_ENCODING, "input G2 point is not in the prime-order subgroup");
    if (fl[0] & 1) return fail(SIPP_ERR_ZERO_CHALLENGE, "challenge is zero: x.inverse().unwrap() panics in the reference");
    if (fl[0] & 2) return fail(SIPP_ERR_ENCODING, "fold scalar recoding failed");
    return SIPP_OK;
}

// The statement tail of a ragged batch, shared by the verifier and the statement prover (verifier_native.rs:74-75, :80): the final
// point of every instance -- its first point once the points are folded -- gathered in the caller's order, paired through the
// products path (one one-pair segment per instance) and encoded.
struct RaggedFinals {
    ProductPlan plan;
    std::vector<uint64_t> at;
    uint32_t *gA = nullptr, *gB = nullptr, *work = nullptr;
    uint64_t* dat = nullptr;
    ProductGroup* dgroups = nullptr;
    ProductTask* dtasks = nullptr;
    ~RaggedFinals() {  // recycled blocks: every caller synchronises its streams before it returns
        pool_free(gA); pool_free(gB); pool_free(work); pool_free(dat); pool_free(dgroups); pool_free(dtasks);
    }
    // the host plan, the device blocks and the line table (before any launch: growing the table frees the old one); offsets checked
    int prepare(const size_t* offsets, size_t count) {
        at.assign(offsets, offsets + count);                                           // final_A = A[0], final_B = B[0]  :74-75
        std::vector<size_t> ones(count + 1);
        for (size_t j = 0; j <= count; j++) ones[j] = j;
        int rc = product_plan(ones.data(), count, g_opt_batch_kpg_max, (size_t)g_opt_product_chunk, plan);
        if (rc) return rc;
        cudaError_t e = pool_alloc((void**)&gA, count * 64);
        if (e == cudaSuccess) e = pool_alloc((void**)&gB, count * 128);
        if (e == cudaSuccess) e = pool_alloc((void**)&work, plan.work_slots(count) * 384);
        if (e == cudaSuccess) e = pool_alloc((void**)&dat, count * sizeof(uint64_t));
        if (e == cudaSuccess) e = pool_alloc((void**)&dgroups, plan.groups.size() * sizeof(ProductGroup));
        if (e == cudaSuccess) e = pool_alloc((void**)&dtasks, plan.tasks.size() * sizeof(ProductTask));
        if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(ragged finals)");
        return lines_reserve((count < plan.chunk_pairs ? count : plan.chunk_pairs) * lines_bytes_per_pair());
    }
    // enqueues on s, after the last fold of dA / dB: pair (when non-NULL) <- count pairings (384 B each, encoded); fin (when non-NULL)
    // <- count x 64 B final_A, then count x 128 B final_B (encoded)
    int run(const uint32_t* dA, const uint32_t* dB, size_t count, uint32_t* pair, uint32_t* fin, cudaStream_t s) {
        if (!pair && !fin) return SIPP_OK;
        CK(cudaMemcpyAsync(dat, at.data(), count * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
        int le = launch_gather_points(dA, dB, dat, count, gA, gB, s);
        if (le) return cuda_fail((cudaError_t)le, "k_gather_points");
        g_stats.launches++;
        if (pair) {                                                                     // pairing(final_A, final_B)  :80
            CK(cudaMemcpyAsync(dgroups, plan.groups.data(), plan.groups.size() * sizeof(ProductGroup), cudaMemcpyHostToDevice, s));
            CK(cudaMemcpyAsync(dtasks, plan.tasks.data(), plan.tasks.size() * sizeof(ProductTask), cudaMemcpyHostToDevice, s));
            le = products_launch(gA, gB, count, count, plan, dgroups, dtasks, work, pair, s);
            if (le) return le;
        }
        if (fin) {
            le = launch_codec_encode(gA, fin, count * 2, s);
            if (!le) le = launch_codec_encode(gB, fin + count * 16, count * 4, s);
            if (le) return cuda_fail((cudaError_t)le, "k_codec_encode");
            g_stats.launches += 2;
        }
        return SIPP_OK;
    }
};

// the whole call: bytesA / bytesB hold the boundary bytes (host staging copies or the caller's device buffers); the proofs are
// copied to `out` (host or device memory, per out_kind) only when every point and every challenge passed its checks.  The statement
// outputs (each may be NULL, then it is not computed): final_A / final_B / final_Z of every instance in the caller's order, copied
// with the proofs.
int ragged_run(const uint32_t* bytesA, const uint32_t* bytesB, size_t n, const size_t* offsets, size_t count, void* out, cudaMemcpyKind out_kind,
               void* final_A, void* final_B, void* final_Z) {
    cudaStream_t s = g_stream;
    RaggedSchedule S;
    int rc = ragged_schedule(offsets, count, S);
    if (rc) return rc;
    const size_t R = S.rounds.size() - 1, act1 = R ? S.rounds[1].act : 0, gather = R ? S.rounds[1].pairs : 0;
    uint32_t *dA = nullptr, *dB = nullptr, *gA = nullptr, *gB = nullptr, *work = nullptr, *res = nullptr, *proofs = nullptr;
    uint64_t *states = nullptr, *ddst = nullptr;
    FoldPlan* plans = nullptr;
    ProductGroup* dgroups = nullptr;
    ProductTask* dtasks = nullptr;
    RaggedInst* dtabs = nullptr;
    RaggedProof* dpt = nullptr;
    int* flags = nullptr;  // [0] transcript / recoding, [1] encoding
    cudaError_t e = pool_alloc((void**)&dA, n * 64);
    if (e == cudaSuccess) e = pool_alloc((void**)&dB, n * 128);
    if (e == cudaSuccess && gather) e = pool_alloc((void**)&gA, gather * 64);
    if (e == cudaSuccess && gather) e = pool_alloc((void**)&gB, gather * 128);
    if (e == cudaSuccess) e = pool_alloc((void**)&work, S.work_slots * 384);
    if (e == cudaSuccess) e = pool_alloc((void**)&res, S.max_products * 384);
    if (e == cudaSuccess) e = pool_alloc((void**)&proofs, S.proof_fq12 * 384);
    if (e == cudaSuccess && act1) e = pool_alloc((void**)&states, act1 * 32);
    if (e == cudaSuccess && act1) e = pool_alloc((void**)&plans, act1 * sizeof(FoldPlan));
    if (e == cudaSuccess) e = pool_alloc((void**)&ddst, S.dst.size() * sizeof(uint64_t));
    if (e == cudaSuccess) e = pool_alloc((void**)&dgroups, S.groups.size() * sizeof(ProductGroup));
    if (e == cudaSuccess) e = pool_alloc((void**)&dtasks, S.tasks.size() * sizeof(ProductTask));
    if (e == cudaSuccess && !S.tabs.empty()) e = pool_alloc((void**)&dtabs, S.tabs.size() * sizeof(RaggedInst));
    if (e == cudaSuccess) e = pool_alloc((void**)&dpt, S.proofs.size() * sizeof(RaggedProof));
    if (e == cudaSuccess) e = pool_alloc((void**)&flags, 2 * sizeof(int));
    struct Release {
        std::vector<void*> p;
        ~Release() { for (void* q : p) pool_free(q); }
    } release{{dA, dB, gA, gB, work, res, proofs, states, plans, ddst, dgroups, dtasks, dtabs, dpt, flags}};  // recycled: later work on s only
    if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(prove_native_batch_ragged)");
    rc = lines_reserve(S.lines_pairs * lines_bytes_per_pair());
    if (rc) return rc;
    RaggedFinals fins;
    uint32_t *pair = nullptr, *enc = nullptr;
    const bool statement = final_A || final_B || final_Z;
    if (statement) {
        rc = fins.prepare(offsets, count);
        if (rc) return rc;
        e = final_Z ? pool_alloc((void**)&pair, count * 384) : cudaSuccess;
        if (e == cudaSuccess && (final_A || final_B)) e = pool_alloc((void**)&enc, count * 192);
        release.p.push_back(pair);
        release.p.push_back(enc);
        if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(prove_native_batch_ragged statement)");
    }
    auto run = [&]() -> int {
        CK(cudaMemsetAsync(flags, 0, 2 * sizeof(int), s));
        CK(cudaMemcpyAsync(ddst, S.dst.data(), S.dst.size() * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(dgroups, S.groups.data(), S.groups.size() * sizeof(ProductGroup), cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(dtasks, S.tasks.data(), S.tasks.size() * sizeof(ProductTask), cudaMemcpyHostToDevice, s));
        if (dtabs) CK(cudaMemcpyAsync(dtabs, S.tabs.data(), S.tabs.size() * sizeof(RaggedInst), cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(dpt, S.proofs.data(), S.proofs.size() * sizeof(RaggedProof), cudaMemcpyHostToDevice, s));
        int le = ragged_decode_absorb(bytesA, bytesB, n, dA, dB, dtabs, act1, states, flags, s);  // round 1's table is the first
        if (le) return le;
        // let Z = inner_product(A, B);  :29 (pushed first)
        const RaggedRound& r0 = S.rounds[0];
        le = products_launch(dA, dB, n, count, r0.plan, dgroups + r0.g0, dtasks + r0.t0, work, res, s);
        if (le) return le;
        le = launch_scatter_fq12(res, ddst + r0.dst0, count, proofs, s);
        if (le) return cuda_fail((cudaError_t)le, "k_scatter_fq12");
        g_stats.launches++;
        for (size_t r = 1; r <= R; r++) {                                                 // :45
            const RaggedRound& rd = S.rounds[r];
            const RaggedInst* tab = dtabs + rd.tab0;
            const unsigned act = (unsigned)rd.act;
            le = launch_ragged_gather(dA, dB, tab, act, rd.elems, gA, gB, s);
            if (le) return cuda_fail((cudaError_t)le, "k_ragged_gather");
            g_stats.launches++;
            le = products_launch(gA, gB, rd.pairs, 2 * rd.act, rd.plan, dgroups + rd.g0, dtasks + rd.t0, work, res, s);  // :46-49
            if (le) return le;
            le = launch_scatter_fq12(res, ddst + rd.dst0, 2 * rd.act, proofs, s);
            if (le) return cuda_fail((cudaError_t)le, "k_scatter_fq12");
            g_stats.launches++;
            {
                Span sp(3, s);
                le = launch_tr_round_ragged(states, proofs, dpt, (int)r, g_opt_fq12_order, act, plans, nullptr, flags, s);  // :42-43 (first round), :52-58
                if (le) return cuda_fail((cudaError_t)le, "k_tr_round_ragged");
                g_stats.launches++;
            }
            {
                Span sp(2, s);
                le = rd.kernel == 2 ? launch_fold_straus_ragged(dA, dB, tab, act, rd.elems, plans, s)
                     : rd.kernel == 1 ? launch_fold_wide_batch_ragged(dA, dB, tab, act, rd.elems, rd.units, plans, s)
                                      : launch_fold_batch_ragged(dA, dB, tab, act, rd.elems, plans, s);  // :60-74
                if (le) return cuda_fail((cudaError_t)le, "k_fold_batch_ragged");
                g_stats.launches++;
                g_stats.fold_points += rd.elems;
            }
        }
        if (statement) {
            le = fins.run(dA, dB, count, pair, enc, s);
            if (le) return le;
        }
        int fl[2] = {0, 0};
        CK(cudaMemcpyAsync(fl, flags, sizeof fl, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        const int st = ragged_flags_status(fl);
        if (st) return st;
        CK(cudaMemcpyAsync(out, proofs, S.proof_fq12 * 384, out_kind, s));
        if (final_A) CK(cudaMemcpyAsync(final_A, enc, count * 64, out_kind, s));
        if (final_B) CK(cudaMemcpyAsync(final_B, enc + count * 16, count * 128, out_kind, s));
        if (final_Z) CK(cudaMemcpyAsync(final_Z, pair, count * 384, out_kind, s));
        CK(cudaStreamSynchronize(s));
        return SIPP_OK;
    };
    rc = run();
    if (rc) cudaStreamSynchronize(s);
    return rc;
}

// the ragged verifier's checks after ragged_args: proof_offsets and results, then the proof lengths (verifier_native.rs:31,40,42)
int ragged_verify_args(const size_t* offsets, size_t count, const size_t* proof_offsets, const int* results) {
    if (!proof_offsets || !results) return fail(SIPP_ERR_ARG, "verify_native_batch_ragged: null pointer");
    if (proof_offsets[0] != 0) return fail(SIPP_ERR_ARG, "verify_native_batch_ragged: proof_offsets[0] != 0");
    for (size_t j = 0; j < count; j++)
        if (proof_offsets[j + 1] < proof_offsets[j]) return fail(SIPP_ERR_ARG, "verify_native_batch_ragged: decreasing proof_offsets");
    for (size_t j = 0; j < count; j++)
        if (proof_offsets[j + 1] - proof_offsets[j] < sipp_proof_len(offsets[j + 1] - offsets[j]))
            return fail(SIPP_ERR_SHORT_PROOF, "proof.pop().unwrap() on an empty proof");
    return SIPP_OK;
}

// where sipp_verify_native_batch_ragged_device wants the outcome: device buffers in the caller's instance order (finals may be NULL)
struct DeviceOutcome {
    int* results;
    uint32_t *final_A, *final_B, *final_Z;
};

// The whole verification on the device (verifier_native.rs:14-85 per instance, every instance in lock-step).  The challenges depend
// only on A, B and the proofs (:33-45), so the transcript is replayed first, round by round over the active instances, and then:
//   main stream  the folds of every round back to back (the prover's fold tables and kernels), the final points gathered in the
//                caller's order and their pairings (:80) through the products path, one one-pair segment per instance;
//   side stream  every GT update in one launch (k_gt_fold_ragged: 1 + log2 n_j factors per instance), one k_seg_product pass
//                (1 + log2 n_j <= 32 <= SIPP_PRODUCT_SPAN factors per instance) and the encode: final_Z of every instance.
// bytesA / bytesB / proofs: boundary bytes in device memory, only read.  Host outcome (dev NULL): out <- count x 384 B final_Z then
// count x 384 B pairings, fin <- count x 64 B final_A then count x 128 B final_B (boundary bytes), copied with the flags.  Device
// outcome: once the flags are clean, k_verify_outcome writes dev's results and finals (of the instances whose proof is canonical).
int ragged_verify_run(const uint32_t* bytesA, const uint32_t* bytesB, size_t n, const size_t* offsets, size_t count, const uint32_t* proofs,
                      const size_t* proof_offsets, uint8_t* out, uint8_t* fin, const DeviceOutcome* dev) {
    cudaStream_t s = g_stream;
    RaggedSchedule S;
    ragged_folds(offsets, count, S);
    const size_t R = S.rounds.size() - 1, act1 = R ? S.rounds[1].act : 0, npow = S.tabs.size();
    // per position k of the order: its proof (the last np_k elements of its slice), its factor slots [fbase[k], fbase[k] + 1 + log2 n_k)
    // -- Z, then the update of round r at fbase[k] + r -- and the task multiplying them into the slot nfac + (caller index)
    std::vector<RaggedProof> pt(count);
    std::vector<RaggedGt> gt(npow + count);
    std::vector<ProductTask> ftasks(count);
    std::vector<size_t> fbase(count);
    size_t nfac = 0;
    for (size_t k = 0; k < count; k++) {
        const size_t j = S.order[k], nj = offsets[j + 1] - offsets[j], np = sipp_proof_len(nj);
        pt[k] = RaggedProof{proof_offsets[j + 1] - np, (uint32_t)np, 0};
        fbase[k] = nfac;
        gt[npow + k] = RaggedGt{pt[k].first + np - 1, (uint32_t)nfac, 0};             // let original_Z = proof.pop().unwrap();  :31
        ftasks[k] = ProductTask{(uint32_t)nfac, (uint32_t)(1 + log2_of(nj)), 0, 0};
        nfac += 1 + log2_of(nj);
    }
    for (size_t k = 0; k < count; k++) ftasks[k].dst = (uint32_t)(nfac + S.order[k]);
    for (size_t r = 1; r <= R; r++)
        for (size_t k = 0; k < S.rounds[r].act; k++)                                   // Z_L at np - 2r, Z_R at np - 1 - 2r  :40, :42
            gt[S.rounds[r].tab0 + k] = RaggedGt{pt[k].first + pt[k].np - 2 * r, (uint32_t)(fbase[k] + r), 0};
    std::vector<RaggedProof> ot(dev ? count : 0);                                     // the device outcome's table: pt in the caller's order
    for (size_t k = 0; k < ot.size(); k++) ot[S.order[k]] = pt[k];
    RaggedFinals fins;
    int rc = fins.prepare(offsets, count);
    if (rc) return rc;
    uint32_t *dA = nullptr, *dB = nullptr, *fac = nullptr;
    uint32_t *res = nullptr, *enc = nullptr;
    uint64_t *states = nullptr, *chal = nullptr;
    FoldPlan* plans = nullptr;
    RaggedInst* dtabs = nullptr;
    RaggedProof *dpt = nullptr, *dot = nullptr;
    RaggedGt* dgt = nullptr;
    ProductTask* dftasks = nullptr;
    int* flags = nullptr;  // [0] transcript / recoding, [1] encoding
    cudaError_t e = pool_alloc((void**)&dA, n * 64);
    if (e == cudaSuccess) e = pool_alloc((void**)&dB, n * 128);
    if (e == cudaSuccess) e = pool_alloc((void**)&fac, (nfac + count) * 384);
    if (e == cudaSuccess) e = pool_alloc((void**)&res, 2 * count * 384);
    if (e == cudaSuccess) e = pool_alloc((void**)&enc, count * 192);
    if (e == cudaSuccess && act1) e = pool_alloc((void**)&states, act1 * 32);
    if (e == cudaSuccess && npow) e = pool_alloc((void**)&chal, npow * 64);
    if (e == cudaSuccess && npow) e = pool_alloc((void**)&plans, npow * sizeof(FoldPlan));
    if (e == cudaSuccess && npow) e = pool_alloc((void**)&dtabs, npow * sizeof(RaggedInst));
    if (e == cudaSuccess) e = pool_alloc((void**)&dpt, count * sizeof(RaggedProof));
    if (e == cudaSuccess) e = pool_alloc((void**)&dgt, gt.size() * sizeof(RaggedGt));
    if (e == cudaSuccess) e = pool_alloc((void**)&dftasks, count * sizeof(ProductTask));
    if (e == cudaSuccess) e = pool_alloc((void**)&flags, 2 * sizeof(int));
    if (e == cudaSuccess && dev) e = pool_alloc((void**)&dot, count * sizeof(RaggedProof));
    struct Release {
        std::vector<void*> p;
        ~Release() { for (void* q : p) pool_free(q); }
    } release{{dA, dB, fac, res, enc, states, chal, plans, dtabs, dpt, dgt, dftasks, flags, dot}};
    if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(verify_native_batch_ragged)");
    if (!g_fold_stream) CK(cudaStreamCreateWithFlags(&g_fold_stream, cudaStreamNonBlocking));
    cudaStream_t side = g_fold_stream;
    bool forked = false;
    auto run = [&]() -> int {
        CK(cudaMemsetAsync(flags, 0, 2 * sizeof(int), s));
        if (npow) CK(cudaMemcpyAsync(dtabs, S.tabs.data(), npow * sizeof(RaggedInst), cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(dpt, pt.data(), count * sizeof(RaggedProof), cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(dgt, gt.data(), gt.size() * sizeof(RaggedGt), cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(dftasks, ftasks.data(), count * sizeof(ProductTask), cudaMemcpyHostToDevice, s));
        if (dev) CK(cudaMemcpyAsync(dot, ot.data(), count * sizeof(RaggedProof), cudaMemcpyHostToDevice, s));
        int le = ragged_decode_absorb(bytesA, bytesB, n, dA, dB, dtabs, act1, states, flags, s);  // round 1's table is the first
        if (le) return le;
        // the transcript replay: round r's fold plans and challenges x || x^-1 to its slices  :33 (first round), :40-46
        for (size_t r = 1; r <= R; r++) {
            const RaggedRound& rd = S.rounds[r];
            Span sp(3, s);
            le = launch_tr_round_ragged(states, proofs, dpt, (int)r, g_opt_fq12_order, (unsigned)rd.act, plans + rd.tab0, chal + 8 * rd.tab0, flags, s);
            if (le) return cuda_fail((cudaError_t)le, "k_tr_round_ragged");
            g_stats.launches++;
        }
        // fork: the GT updates (:59-61) need the proofs and the challenges only
        CK(order_after(side, s));
        forked = true;
        {
            Span sp(1, side);
            le = launch_gt_fold_ragged(proofs, dgt, npow, count, chal, fac, side);
            if (le) return cuda_fail((cudaError_t)le, "k_gt_fold_ragged");
            le = launch_seg_product(dftasks, count, fac, side);
            if (le) return cuda_fail((cudaError_t)le, "k_seg_product");
            le = launch_reduce_fe_eng(fac + nfac * 96, 1, (int)count, res, 2, g_opt_fe_norm, side);  // product + encode
            if (le) return cuda_fail((cudaError_t)le, "k_reduce_fe_eng");
            g_stats.launches += 3;
        }
        for (size_t r = 1; r <= R; r++) {                                                 // :35
            const RaggedRound& rd = S.rounds[r];
            const RaggedInst* tab = dtabs + rd.tab0;
            const FoldPlan* pl = plans + rd.tab0;
            const unsigned act = (unsigned)rd.act;
            Span sp(2, s);
            const int le = rd.kernel == 2 ? launch_fold_straus_ragged(dA, dB, tab, act, rd.elems, pl, s)
                           : rd.kernel == 1 ? launch_fold_wide_batch_ragged(dA, dB, tab, act, rd.elems, rd.units, pl, s)
                                            : launch_fold_batch_ragged(dA, dB, tab, act, rd.elems, pl, s);  // :48-57
            if (le) return cuda_fail((cudaError_t)le, "k_fold_batch_ragged");
            g_stats.launches++;
            g_stats.fold_points += rd.elems;
        }
        le = fins.run(dA, dB, count, res + count * 96, enc, s);                         // :74-75, :80
        if (le) return le;
        CK(order_after(s, side));  // join
        int fl[2] = {0, 0};
        CK(cudaMemcpyAsync(fl, flags, sizeof fl, cudaMemcpyDeviceToHost, s));
        if (!dev) {
            CK(cudaMemcpyAsync(out, res, 2 * count * 384, cudaMemcpyDeviceToHost, s));
            CK(cudaMemcpyAsync(fin, enc, count * 192, cudaMemcpyDeviceToHost, s));
        }
        CK(cudaStreamSynchronize(s));
        const int st = ragged_flags_status(fl);
        if (st || !dev) return st;
        le = launch_verify_outcome(proofs, dot, count, res, res + count * 96, enc, false, dev->results, dev->final_A, dev->final_B, dev->final_Z, s);
        if (le) return cuda_fail((cudaError_t)le, "k_verify_outcome");
        g_stats.launches++;
        CK(cudaStreamSynchronize(s));
        return SIPP_OK;
    };
    rc = run();
    if (rc) {  // neither stream may still use a block when the pool recycles it
        if (forked) order_after(s, side);
        cudaStreamSynchronize(side);
        cudaStreamSynchronize(s);
    }
    return rc;
}

}  // namespace

extern "C" {

int sipp_prove_native_batch_ragged_statement(const uint8_t* A, size_t a_len, const uint8_t* B, size_t b_len, const size_t* offsets, size_t count,
                                             uint8_t* proofs, uint8_t* final_A, uint8_t* final_B, uint8_t* final_Z) {
    int rc = ragged_args(A, a_len, B, b_len, offsets, count, proofs);
    if (rc) return rc;
    rc = ensure_init();
    if (rc) return rc;
    uint32_t *tA = nullptr, *tB = nullptr;
    cudaError_t e = pool_alloc((void**)&tA, a_len * 64);
    if (e == cudaSuccess) e = pool_alloc((void**)&tB, a_len * 128);
    struct Release {
        uint32_t *a, *b;
        ~Release() { pool_free(a); pool_free(b); }
    } release{tA, tB};
    if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(prove_native_batch_ragged)");
    CK(cudaMemcpyAsync(tA, A, a_len * 64, cudaMemcpyHostToDevice, g_stream));
    CK(cudaMemcpyAsync(tB, B, a_len * 128, cudaMemcpyHostToDevice, g_stream));
    return ragged_run(tA, tB, a_len, offsets, count, proofs, cudaMemcpyDeviceToHost, final_A, final_B, final_Z);  // synchronises
}

int sipp_prove_native_batch_ragged_statement_device(const void* dA, const void* dB, size_t n, const size_t* offsets, size_t count, void* d_proofs,
                                                    void* d_final_A, void* d_final_B, void* d_final_Z) {
    int rc = ragged_args(dA, n, dB, n, offsets, count, d_proofs);
    if (rc) return rc;
    rc = ensure_init();
    if (rc) return rc;
    return ragged_run((const uint32_t*)dA, (const uint32_t*)dB, n, offsets, count, d_proofs, cudaMemcpyDeviceToDevice, d_final_A, d_final_B, d_final_Z);
}

int sipp_prove_native_batch_ragged(const uint8_t* A, size_t a_len, const uint8_t* B, size_t b_len, const size_t* offsets, size_t count, uint8_t* proofs) {
    return sipp_prove_native_batch_ragged_statement(A, a_len, B, b_len, offsets, count, proofs, nullptr, nullptr, nullptr);
}

int sipp_prove_native_batch_ragged_device(const void* dA, const void* dB, size_t n, const size_t* offsets, size_t count, void* d_proofs) {
    return sipp_prove_native_batch_ragged_statement_device(dA, dB, n, offsets, count, d_proofs, nullptr, nullptr, nullptr);
}

int sipp_verify_native_batch_ragged(const uint8_t* A, size_t a_len, const uint8_t* B, size_t b_len, const size_t* offsets, size_t count,
                                    const uint8_t* proofs, const size_t* proof_offsets, int* results, uint8_t* final_A, uint8_t* final_B,
                                    uint8_t* final_Z) {
    int rc = ragged_args(A, a_len, B, b_len, offsets, count, proofs);
    if (rc) return rc;
    rc = ragged_verify_args(offsets, count, proof_offsets, results);
    if (rc) return rc;
    rc = ensure_init();
    if (rc) return rc;
    std::vector<uint8_t> out(2 * count * 384), fin(count * 192);
    {
        const size_t ptotal = proof_offsets[count];
        uint32_t *bA = nullptr, *bB = nullptr, *dproofs = nullptr;
        cudaError_t e = pool_alloc((void**)&bA, a_len * 64);
        if (e == cudaSuccess) e = pool_alloc((void**)&bB, a_len * 128);
        if (e == cudaSuccess) e = pool_alloc((void**)&dproofs, ptotal * 384);
        struct Release {
            uint32_t *a, *b, *p;
            ~Release() { pool_free(a); pool_free(b); pool_free(p); }
        } release{bA, bB, dproofs};  // recycled: later work on g_stream only
        if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(verify_native_batch_ragged)");
        CK(cudaMemcpyAsync(bA, A, a_len * 64, cudaMemcpyHostToDevice, g_stream));
        CK(cudaMemcpyAsync(bB, B, a_len * 128, cudaMemcpyHostToDevice, g_stream));
        CK(cudaMemcpyAsync(dproofs, proofs, ptotal * 384, cudaMemcpyHostToDevice, g_stream));
        rc = ragged_verify_run(bA, bB, a_len, offsets, count, dproofs, proof_offsets, out.data(), fin.data(), nullptr);
    }
    if (rc) return rc;
    for (size_t j = 0; j < count; j++) {
        // a proof with a coordinate >= p is one the reference could not have deserialised: refused on its own, like a bad A or B
        const size_t np = sipp_proof_len(offsets[j + 1] - offsets[j]);
        if (!fq_bytes_canonical(proofs + 384 * (proof_offsets[j + 1] - np), 12 * np)) {
            results[j] = SIPP_ERR_ENCODING;
            continue;
        }
        results[j] = memcmp(&out[384 * j], &out[384 * (count + j)], 384) == 0 ? SIPP_OK : SIPP_ERR_VERIFY;  // :81-84
        if (final_A) memcpy(final_A + 64 * j, &fin[64 * j], 64);
        if (final_B) memcpy(final_B + 128 * j, &fin[64 * count + 128 * j], 128);
        if (final_Z) memcpy(final_Z + 384 * j, &out[384 * j], 384);
    }
    return SIPP_OK;
}

int sipp_verify_native_batch_ragged_device(const void* dA, const void* dB, size_t n, const size_t* offsets, size_t count, const void* d_proofs,
                                           const size_t* proof_offsets, int* d_results, void* d_final_A, void* d_final_B, void* d_final_Z) {
    int rc = ragged_args(dA, n, dB, n, offsets, count, d_proofs);
    if (rc) return rc;
    rc = ragged_verify_args(offsets, count, proof_offsets, d_results);
    if (rc) return rc;
    rc = ensure_init();
    if (rc) return rc;
    CK(order_after(g_stream, cudaStreamLegacy));  // inputs just written on the legacy default stream (torch's, unless switched)
    const DeviceOutcome dev{d_results, (uint32_t*)d_final_A, (uint32_t*)d_final_B, (uint32_t*)d_final_Z};
    return ragged_verify_run((const uint32_t*)dA, (const uint32_t*)dB, n, offsets, count, (const uint32_t*)d_proofs, proof_offsets, nullptr, nullptr,
                             &dev);
}

// host-only schedule of a ragged batch (no GPU needed) under the current options: 5 words per round r = 0 .. log2 max n_j -- active
// instances, pairs, fold elements, fold kernel (-1 none, 0 k_fold_batch, 1 k_fold_wide_batch, 2 k_fold_straus) and line-table
// chunks -- to `out` when out_cap >= 5 x rounds; returns the number of rounds or a negative status
long sipp_test_ragged_schedule(const size_t* offsets, size_t count, long long* out, size_t out_cap) {
    if (!offsets) return fail(SIPP_ERR_ARG, "null offsets");
    int rc = ragged_args(offsets, offsets[count], offsets, offsets[count], offsets, count, offsets);
    if (rc) return rc;
    RaggedSchedule S;
    rc = ragged_schedule(offsets, count, S);
    if (rc) return rc;
    const size_t rounds = S.rounds.size();
    if (out && out_cap >= 5 * rounds) {
        for (size_t r = 0; r < rounds; r++) {
            const RaggedRound& rd = S.rounds[r];
            out[5 * r] = (long long)rd.act;
            out[5 * r + 1] = (long long)rd.pairs;
            out[5 * r + 2] = (long long)rd.elems;
            out[5 * r + 3] = rd.kernel;
            out[5 * r + 4] = (long long)rd.plan.chunks();
        }
    }
    return (long)rounds;
}

}  // extern "C"

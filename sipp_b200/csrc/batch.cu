// batch.cu -- batched instances: `count` independent SIPP instances proved (and verified) in lock-step (C ABI: sipp_prove_native_batch,
// sipp_prove_native_batch_device, sipp_verify_native_batch; BASELINE config "4096 independent n=128 SIPP instances").
//
// `count` independent SIPP instances of n pairs each, proved in lock-step: round k of every instance runs in the same launches
// (BASELINE config "4096 independent n=128 SIPP instances").  Each instance is exactly sipp_prove_native (prover_native.rs:26-80);
// what changes is where the glue runs: one transcript chain per instance on the device (k_transcript.cu), per-instance fold
// plans, segmented products.  Nothing returns to the host between the upload and the proofs.
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "host_state.h"

using namespace sipp;
using namespace sipp_host;

namespace {

struct BatchBuffers {
    uint32_t *bytesA = nullptr, *bytesB = nullptr;  // boundary bytes (the transcript reads canonical limbs)
    uint32_t *dA = nullptr, *dB = nullptr;          // Montgomery
    uint32_t* proofs = nullptr;                     // [count][np][96]
    uint32_t* partials = nullptr;
    uint64_t* states = nullptr;
    FoldPlan* plans = nullptr;
    int* flags = nullptr;                           // [0] transcript / recoding, [1] encoding
    void release() {
        pool_free(bytesA); pool_free(bytesB); pool_free(dA); pool_free(dB); pool_free(proofs); pool_free(partials);
        pool_free(states); pool_free(plans); pool_free(flags);
    }
};

size_t pow2_floor(size_t v) {
    size_t r = 1;
    while (r * 2 <= v) r *= 2;
    return r;
}

// products of the current round of every instance: which = 0 -> Z (slot0), which = 1 -> Z_L (slot0), Z_R (slot1)
// `lines` / `lines_cap`: this caller's slice of the process line table (sub-batches on different streams use disjoint slices)
// `qlines` (or NULL): Q-only line coefficients of every B point of the slice (k_qlines_batch), valid while B is unfolded
int batch_products(const BatchBuffers& b, size_t stride, size_t count, size_t m, int which, uint32_t* fe_out, size_t np, int slot0, int slot1, uint32_t* lines,
                   size_t lines_cap, const uint32_t* qlines, cudaStream_t s) {
    BatchJob job;
    job.stride = stride;
    if (which == 0) {
        job.nprod = 1; job.h = m;
        job.a_off[0] = job.b_off[0] = job.a_off[1] = job.b_off[1] = 0;
    } else {
        job.nprod = 2; job.h = m / 2;
        job.a_off[0] = job.h; job.b_off[0] = 0;   // Z_L = inner_product(A2, B1)   prover_native.rs:48
        job.a_off[1] = 0; job.b_off[1] = job.h;   // Z_R = inner_product(A1, B2)   prover_native.rs:49
    }
    const size_t nproducts = count * (size_t)job.nprod;
    const size_t per_pair = lines_bytes_per_pair();
    size_t pc = lines_cap / (job.h * per_pair);  // products per chunk (whole products only)
    if (pc < 1) return fail(SIPP_ERR_ARG, "batched instances: one product exceeds the line buffer (use sipp_prove_native for large n)");
    if (pc > nproducts) pc = nproducts;
    // accumulator groups: kpg pairs of ONE product share an accumulator and its 64 squarings (5,070 Fq-mul-eq per group, 3,661
    // per pair).  The GPU holds 2 blocks x 20 groups per SM at a time; pick the power of two that minimises waves x group length.
    size_t kpg = 1;
    {
        const size_t wave = (size_t)g_sm_count * 40;
        double best = 0;
        for (size_t cand = 1; cand <= job.h && cand <= (size_t)g_opt_batch_kpg_max; cand *= 2) {
            if (job.h % cand) break;  // h is a power of two in a proof; any h still works with kpg = 1
            size_t groups = pc * job.h / cand;
            double cost = (double)((groups + wave - 1) / wave) * (5070.0 + 3661.0 * (double)cand);
            if (best == 0 || cost < best) { best = cost; kpg = cand; }
        }
    }
    const size_t gpp = job.h / kpg;
    {
        Span sp(0, s);
        for (size_t p0 = 0; p0 < nproducts; p0 += pc) {
            size_t cur = nproducts - p0 < pc ? nproducts - p0 : pc;
            // shared coefficients (Z, first cross products) / 16 lanes per pair for a launch that cannot fill the GPU / one thread per pair
            int e = qlines ? launch_eval_lines_batch(b.dA, b.dB, job, p0, cur, qlines, lines, s)
                    : cur * job.h <= (size_t)g_opt_wide_max ? launch_lines_wide_batch(b.dA, b.dB, job, p0, cur, lines, s)
                                                            : launch_lines_batch(b.dA, b.dB, job, p0, cur, lines, s);
            if (e) return cuda_fail((cudaError_t)e, "k_lines_batch");
            e = launch_accum_batch(lines, cur * job.h, (int)kpg, b.partials, p0 * gpp, s);
            if (e) return cuda_fail((cudaError_t)e, "k_accum(batch)");
            g_stats.launches += 2;
            g_stats.miller_launches++;
        }
    }
    g_stats.miller_pairs += nproducts * job.h;
    {
        Span sp(1, s);
        // one 32-lane machine per product while they all fit the GPU at once (3 blocks x 4 machines per SM), 6-lane groups beyond
        int e = (g_opt_fe_engine && nproducts <= (size_t)g_sm_count * 12)
                    ? launch_fe_batch_eng(b.partials, nproducts, (int)gpp, job.nprod, fe_out, np * 96, slot0, slot1, g_opt_fe_norm, s)
                    : launch_fe_batch(b.partials, nproducts, (int)gpp, job.nprod, fe_out, np * 96, slot0, slot1, g_opt_fe_norm, s);
        if (e) return cuda_fail((cudaError_t)e, "k_fe_batch");
    }
    g_stats.launches++;
    return SIPP_OK;
}

// line-table budget of one batched call, split evenly over its sub-batches
const size_t kBatchLinesCap = (size_t)16 << 30;

// slice [i0, i0 + c) of the instances of a batch
BatchBuffers batch_view(const BatchBuffers& b, size_t n, size_t np, size_t i0) {
    BatchBuffers v = b;
    v.bytesA = b.bytesA + i0 * n * 16; v.bytesB = b.bytesB + i0 * n * 32;
    v.dA = b.dA + i0 * n * 16; v.dB = b.dB + i0 * n * 32;
    v.proofs = b.proofs ? b.proofs + i0 * np * 96 : nullptr;
    v.partials = b.partials + i0 * n * 96;
    v.states = b.states + i0 * 4;
    v.plans = b.plans + i0;
    return v;
}

// Sub-batches (SIPP_OPT_BATCH_STREAMS, off by default): the late rounds of a batch are latency-bound (a launch of a few thousand
// pairs does not fill 148 SMs), so a batch can be cut into independent sub-batches on their own streams whose kernels run side by
// side.  Measured: no gain (see batch_sub_count) -- kept as an experiment switch.
int g_sub_streams_dev = -1;
cudaStream_t g_sub_streams[8];
int batch_sub_count(size_t n, size_t count) {
    if (g_opt_profile) return 1;  // per-kernel-class event spans are only meaningful when the launches do not overlap
    int want = g_opt_batch_streams;
    if (want <= 0) want = 1;  // measured on B200 (512 and 4096 instances of n = 128): 1 / 2 / 4 / 8 sub-batches = 95 / 98 / 104 / 103 ms and
                              // 401 / 398 / 423 / 460 ms -- concurrent sub-batches run in the same phase and compete, so the default is one
    if (want > 8) want = 8;
    while (want > 1 && count / (size_t)want < 32) want /= 2;
    return want < 1 ? 1 : want;
}

// the whole batch on the device; bytesA / bytesB already hold the boundary bytes.  Enqueues everything; the caller synchronises.
cudaStream_t g_side = nullptr;  // transcript absorb chains of a large batch, next to the first products
int g_side_dev = -1;
}  // namespace
namespace sipp_host {
// sipp_shutdown / a device switch: the per-device streams of the batched prover
void batch_release_streams() {
    if (g_side_dev >= 0 && g_side) cudaStreamDestroy(g_side);
    g_side = nullptr;
    g_side_dev = -1;
    if (g_sub_streams_dev >= 0)
        for (int k = 0; k < 8; k++) cudaStreamDestroy(g_sub_streams[k]);
    g_sub_streams_dev = -1;
}
}  // namespace sipp_host
namespace {

int batch_prove_enqueue(BatchBuffers& b, size_t n, size_t count, cudaStream_t s, bool* side_used, int* subs_used);
int batch_prove_resident(BatchBuffers& b, size_t n, size_t count, cudaStream_t s) {
    bool side_used = false;
    int subs_used = 0;
    const int rc = batch_prove_enqueue(b, n, count, s, &side_used, &subs_used);
    // whatever happened (an error return in the middle of a round included), `s` must not run ahead of the side stream and the
    // sub-batch streams: the caller synchronises `s` only and then recycles the buffers they may still be using
    if (side_used) order_after(s, g_side);
    for (int k = 0; k < subs_used; k++) order_after(s, g_sub_streams[k]);
    return rc;
}

int batch_prove_enqueue(BatchBuffers& b, size_t n, size_t count, cudaStream_t s, bool* side_used, int* subs_used) {
    const size_t np = sipp_proof_len(n), total = n * count;
    CK(cudaMemsetAsync(b.flags, 0, 2 * sizeof(int), s));
    {
        Span sp(3, s);
        int e = launch_codec_decode(b.bytesA, b.dA, total * 2, b.flags + 1, s);
        if (!e) e = launch_codec_decode(b.bytesB, b.dB, total * 4, b.flags + 1, s);
        if (e) return cuda_fail((cudaError_t)e, "k_codec_decode");
        g_stats.launches += 2;
        if (g_opt_validate) {  // on the curve, B_i in the order-r subgroup (SIPP_OPT_VALIDATE_POINTS)
            e = launch_validate_points(b.dA, b.dB, total, b.flags + 1, s);
            if (e) return cuda_fail((cudaError_t)e, "k_validate_points");
            g_stats.launches++;
        }
    }
    // register A and B (prover_native.rs:36-39): independent of everything the products compute, so the chains run on a side
    // stream next to Z and the first Z_L, Z_R
    if (g_side_dev != g_device) {
        CK(cudaStreamCreateWithFlags(&g_side, cudaStreamNonBlocking));
        g_side_dev = g_device;
    }
    cudaStream_t side = g_side;
    if (g_sub_streams_dev != g_device) {
        for (int k = 0; k < 8; k++) CK(cudaStreamCreateWithFlags(&g_sub_streams[k], cudaStreamNonBlocking));
        g_sub_streams_dev = g_device;
    }
    // small batches: the chains are latency-bound and slow down several times when they share the SMs with the Miller kernels,
    // which then wait for them at the first challenge -- run them first, alone (SIPP_BATCH_ABSORB=side|inline overrides)
    static const char* absorb_env = getenv("SIPP_BATCH_ABSORB");
    const bool absorb_inline = absorb_env ? absorb_env[0] == 'i' : total < ((size_t)1 << 18);
    cudaStream_t absorb_stream = absorb_inline ? s : side;
    if (!absorb_inline) {
        CK(order_after(side, s));
        *side_used = true;
    }
    {
        Span sp(3, absorb_stream);
        int e = launch_tr_absorb_pairs(b.bytesA, b.bytesB, n, count, b.states, absorb_stream);
        if (e) return cuda_fail((cudaError_t)e, "k_tr_absorb_pairs");
        g_stats.launches++;
    }
    const int nsub = batch_sub_count(n, count);
    // line table: every sub-batch gets a slice large enough for its largest launch (Z: all n pairs of its instances), within the budget
    const size_t per_pair = lines_bytes_per_pair();
    const size_t sub_max = (count + nsub - 1) / nsub;
    size_t slice = sub_max * n * per_pair;
    if (slice > kBatchLinesCap / nsub) slice = kBatchLinesCap / nsub;
    slice = (slice + 255) & ~(size_t)255;
    int rc = lines_reserve(slice * nsub);
    if (rc) return rc;
    // Q-only line coefficients of all B points, when they fit the budget (17,472 B per point)
    uint32_t* qbuf = nullptr;
    if (g_opt_batch_qlines && total * qlines_bytes_per_point() <= kBatchLinesCap) {
        cudaError_t qe = pool_alloc((void**)&qbuf, total * qlines_bytes_per_point());
        if (qe != cudaSuccess) return cuda_fail(qe, "cudaMalloc(qlines)");
    }
    struct QFree { uint32_t* p; ~QFree() { pool_free(p); } } qfree{qbuf};  // recycled block: later work on the same streams only
    // fork: every sub-stream waits for the decode on `s` (ordered BEFORE any join below, or sub-batch k + 1 would wait for k)
    for (int k = 0; k < nsub && nsub > 1; k++) CK(order_after(g_sub_streams[k], s));
    *subs_used = nsub > 1 ? nsub : 0;
    for (int k = 0; k < nsub; k++) {
        const size_t i0 = count * (size_t)k / nsub, i1 = count * (size_t)(k + 1) / nsub, c = i1 - i0;
        if (c == 0) continue;
        cudaStream_t sk = nsub == 1 ? s : g_sub_streams[k];
        BatchBuffers v = batch_view(b, n, np, i0);
        uint32_t* lines = lines_buffer() + (slice / 4) * k;
        // every B_i is paired twice before the first fold (in Z and in the first Z_L / Z_R): walk it through the schedule once
        const uint32_t* ql = nullptr;
        if (qbuf && n >= 2) {
            uint32_t* q = qbuf + i0 * n * (qlines_bytes_per_point() / 4);
            Span sp(0, sk);
            int e = launch_qlines_batch(v.dB, c * n, q, sk);
            if (e) return cuda_fail((cudaError_t)e, "k_qlines_batch");
            g_stats.launches++;
            ql = q;
        }
        rc = batch_products(v, n, c, n, 0, v.proofs, np, (int)np - 1, 0, lines, slice, ql, sk);   // let Z = inner_product(A, B);  :29 (pushed first)
        if (rc) return rc;
        size_t m = n;
        int round = 1;
        while (m > 1) {                                                            // :45
            const int slot_l = (int)np - 2 * round, slot_r = (int)np - 1 - 2 * round;  // proof.reverse()  :78
            rc = batch_products(v, n, c, m, 1, v.proofs, np, slot_l, slot_r, lines, slice, round == 1 ? ql : nullptr, sk);  // :46-49
            if (rc) return rc;
            if (round == 1 && !absorb_inline) CK(order_after(sk, side));
            {
                Span sp(3, sk);
                int e = launch_tr_round(v.states, v.proofs, np, round == 1 ? (int)np - 1 : -1, slot_l, slot_r, g_opt_fq12_order, c, v.plans, nullptr,
                                        b.flags, sk);                              // :42-43 (first round), :52-58
                if (e) return cuda_fail((cudaError_t)e, "k_tr_round");
                g_stats.launches++;
            }
            {
                Span sp(2, sk);
                // one thread per element (shared doublings) when the launch fills the GPU; otherwise the lane-split components, whose
                // dependent chain is 3x shorter when a warp spans several instances (divergent digit tests)
                const size_t elems = c * (m / 2);
                int e = (g_opt_fold_straus && elems >= 16384)          ? launch_fold_straus(v.dA, v.dB, m / 2, n, c, v.plans, sk)
                        : elems <= (size_t)g_opt_wide_fold_max + 512   ? launch_fold_wide_batch(v.dA, v.dB, m / 2, n, c, v.plans, sk)  // lane engine: <= 2 waves
                                                                       : launch_fold_batch(v.dA, v.dB, m / 2, n, c, v.plans, sk);      // :60-74
                if (e) return cuda_fail((cudaError_t)e, "k_fold_batch");
                g_stats.launches++;
                g_stats.fold_points += c * (m / 2);
            }
            m /= 2;
            round++;
        }
    }
    return SIPP_OK;  // the caller (batch_prove_resident) joins the side stream and the sub-streams into `s`
}

int batch_alloc(BatchBuffers& b, size_t n, size_t count) {
    const size_t np = sipp_proof_len(n), total = n * count;
    // worst case one accumulator group per pair
    cudaError_t e = pool_alloc((void**)&b.bytesA, total * 64);
    if (e == cudaSuccess) e = pool_alloc((void**)&b.bytesB, total * 128);
    if (e == cudaSuccess) e = pool_alloc((void**)&b.dA, total * 64);
    if (e == cudaSuccess) e = pool_alloc((void**)&b.dB, total * 128);
    if (e == cudaSuccess) e = pool_alloc((void**)&b.proofs, count * np * 384);
    if (e == cudaSuccess) e = pool_alloc((void**)&b.partials, total * 384);
    if (e == cudaSuccess) e = pool_alloc((void**)&b.states, count * 32);
    if (e == cudaSuccess) e = pool_alloc((void**)&b.plans, count * sizeof(FoldPlan));
    if (e == cudaSuccess) e = pool_alloc((void**)&b.flags, 2 * sizeof(int));
    if (e != cudaSuccess) {
        b.release();
        return cuda_fail(e, "cudaMalloc(batch)");
    }
    return SIPP_OK;
}

int batch_check_flags(const BatchBuffers& b, cudaStream_t s) {
    int flags[2] = {0, 0};
    CK(cudaMemcpyAsync(flags, b.flags, sizeof flags, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    if (flags[1] & 1) return fail(SIPP_ERR_ENCODING, "input coordinate >= p");
    if (flags[1] & 2) return fail(SIPP_ERR_ENCODING, "input point is not on the curve");
    if (flags[1] & 4) return fail(SIPP_ERR_ENCODING, "input G2 point is not in the prime-order subgroup");
    if (flags[0] & 1) return fail(SIPP_ERR_ZERO_CHALLENGE, "challenge is zero: x.inverse().unwrap() panics in the reference");
    if (flags[0] & 2) return fail(SIPP_ERR_ENCODING, "fold scalar recoding failed");
    return SIPP_OK;
}

// The statement members of every instance once its points are folded to one, A[0] and B[0] (verifier_native.rs:74-75): to `pair`
// (when non-NULL) pairing(final_A, final_B) of every instance (:80; count x 384 B, encoded), to `fin` (when non-NULL) final_A
// (count x 64 B) then final_B (count x 128 B), encoded.  Reuses b.bytesA / b.bytesB, which the rounds no longer read.
int batch_finals(const BatchBuffers& b, size_t n, size_t count, uint32_t* pair, uint32_t* fin, cudaStream_t s) {
    if (pair) {
        int rc = lines_reserve(count * lines_bytes_per_pair());
        if (rc) return rc;
        rc = batch_products(b, n, count, 1, 0, pair, 1, 0, 0, lines_buffer(), count * lines_bytes_per_pair(), nullptr, s);
        if (rc) return rc;
    }
    if (fin) {
        CK(cudaMemcpy2DAsync(b.bytesA, 64, b.dA, n * 64, 64, count, cudaMemcpyDeviceToDevice, s));
        CK(cudaMemcpy2DAsync(b.bytesB, 128, b.dB, n * 128, 128, count, cudaMemcpyDeviceToDevice, s));
        int le = launch_codec_encode(b.bytesA, fin, count * 2, s);
        if (!le) le = launch_codec_encode(b.bytesB, fin + count * 16, count * 4, s);
        if (le) return cuda_fail((cudaError_t)le, "batch finals: encode");
        g_stats.launches += 2;
    }
    return SIPP_OK;
}

int batch_args(const void* A, const void* B, size_t n, size_t count, const void* proofs) {
    if (!A || !B || !proofs || count == 0) return fail(SIPP_ERR_ARG, "null pointer or count == 0");
    if (!is_pow2(n)) return fail(SIPP_ERR_ARG, "n must be a non-zero power of two");
    return SIPP_OK;
}

// The device blocks of a batched verification.  staging: the host form uploads A, B and the proofs to b.bytesA, b.bytesB and
// dproofs; otherwise b.bytesA / b.bytesB are only the scratch of batch_finals (count points each) and there is no dproofs.
struct VerifyBuffers {
    BatchBuffers b;
    uint32_t *dproofs = nullptr, *dz = nullptr, *dpair = nullptr, *dfin = nullptr;
    uint64_t* dchal = nullptr;
    int alloc(size_t n, size_t count, size_t proof_len, bool staging) {
        const size_t pts = staging ? n * count : count, total = n * count;
        cudaError_t e = pool_alloc((void**)&b.bytesA, pts * 64);
        if (e == cudaSuccess) e = pool_alloc((void**)&b.bytesB, pts * 128);
        if (e == cudaSuccess) e = pool_alloc((void**)&b.dA, total * 64);
        if (e == cudaSuccess) e = pool_alloc((void**)&b.dB, total * 128);
        if (e == cudaSuccess) e = pool_alloc((void**)&b.partials, count * 384);
        if (e == cudaSuccess) e = pool_alloc((void**)&b.states, count * 32);
        if (e == cudaSuccess) e = pool_alloc((void**)&b.plans, count * sizeof(FoldPlan));
        if (e == cudaSuccess) e = pool_alloc((void**)&b.flags, 2 * sizeof(int));
        if (e == cudaSuccess && staging) e = pool_alloc((void**)&dproofs, count * proof_len * 384);
        if (e == cudaSuccess) e = pool_alloc((void**)&dz, count * 384);
        if (e == cudaSuccess) e = pool_alloc((void**)&dpair, count * 384);
        if (e == cudaSuccess) e = pool_alloc((void**)&dfin, count * 192);
        if (e == cudaSuccess) e = pool_alloc((void**)&dchal, count * 64);
        return e == cudaSuccess ? SIPP_OK : cuda_fail(e, "cudaMalloc(verify batch)");
    }
    ~VerifyBuffers() {  // recycled blocks: every caller synchronises the stream before it returns
        b.release();
        pool_free(dproofs); pool_free(dz); pool_free(dpair); pool_free(dfin); pool_free(dchal);
    }
};

// `count` independent verifications in lock-step (verifier_native.rs:14-80 per instance) on boundary bytes in device memory, which are
// only read: bytesA / bytesB (count x n points), proofs (count x proof_len Fq12).  The transcript replay, the folds and the GT update
// Z_L^x Z Z_R^(x^-1) of every instance run in the same launches; the final pairing check (:80) is one batched product of one pair per
// instance.  Enqueues on s: final_Z to v.dz, the pairings to v.dpair and, when fin, final_A then final_B to v.dfin (encoded).
int batch_verify_enqueue(VerifyBuffers& v, const uint32_t* bytesA, const uint32_t* bytesB, const uint32_t* proofs, size_t n, size_t count,
                         size_t proof_len, bool fin, cudaStream_t s) {
    BatchBuffers& b = v.b;
    const size_t total = n * count, top = proof_len;  // the verifier pops from the end: Z = proof[top - 1]
    CK(cudaMemsetAsync(b.flags, 0, 2 * sizeof(int), s));
    int le = launch_codec_decode(bytesA, b.dA, total * 2, b.flags + 1, s);
    if (!le) le = launch_codec_decode(bytesB, b.dB, total * 4, b.flags + 1, s);
    if (!le && g_opt_validate) { le = launch_validate_points(b.dA, b.dB, total, b.flags + 1, s); g_stats.launches++; }
    if (!le) le = launch_tr_absorb_pairs(bytesA, bytesB, n, count, b.states, s);                       // :25-28
    if (le) return cuda_fail((cudaError_t)le, "verify batch: decode / absorb");
    g_stats.launches += 3;
    // let original_Z = proof.pop().unwrap();  :31   (Z of instance j = its last Fq12)
    CK(cudaMemcpy2DAsync(v.dz, 384, (const uint8_t*)proofs + (top - 1) * 384, proof_len * 384, 384, count, cudaMemcpyDeviceToDevice, s));
    size_t m = n;
    int round = 1;
    while (m > 1) {                                                                                     // :35
        const int slot_l = (int)top - 2 * round, slot_r = (int)top - 1 - 2 * round;                     // :40, :42
        le = launch_tr_round(b.states, proofs, proof_len, round == 1 ? (int)top - 1 : -1, slot_l, slot_r, g_opt_fq12_order, count, b.plans,
                             v.dchal, b.flags, s);                                                       // :33 (first round), :41-46
        if (!le) le = (g_opt_fold_straus && count * (m / 2) >= 16384) ? launch_fold_straus(b.dA, b.dB, m / 2, n, count, b.plans, s)
                                                                         : launch_fold_batch(b.dA, b.dB, m / 2, n, count, b.plans, s);  // :48-57
        if (!le) le = launch_gt_fold_batch(proofs, proof_len, slot_l, slot_r, v.dchal, v.dz, count, s);  // :59-61
        if (le) return cuda_fail((cudaError_t)le, "verify batch: round");
        g_stats.launches += 3;
        g_stats.fold_points += count * (m / 2);
        m /= 2;
        round++;
    }
    return batch_finals(b, n, count, v.dpair, fin ? v.dfin : nullptr, s);                              // :74-75, :80
}

}  // namespace

extern "C" {

int sipp_prove_native_batch_device(const void* dA, const void* dB, size_t n, size_t count, void* d_proofs) {
    int rc = ensure_init();
    if (rc) return rc;
    rc = batch_args(dA, dB, n, count, d_proofs);
    if (rc) return rc;
    const size_t np = sipp_proof_len(n);
    BatchBuffers b;
    rc = batch_alloc(b, n, count);
    if (rc) return rc;
    cudaError_t e = cudaMemcpyAsync(b.bytesA, dA, n * count * 64, cudaMemcpyDeviceToDevice, g_stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(b.bytesB, dB, n * count * 128, cudaMemcpyDeviceToDevice, g_stream);
    if (e != cudaSuccess) { b.release(); return cuda_fail(e, "D2D"); }
    rc = batch_prove_resident(b, n, count, g_stream);
    if (!rc) {
        e = cudaMemcpyAsync(d_proofs, b.proofs, count * np * 384, cudaMemcpyDeviceToDevice, g_stream);
        if (e != cudaSuccess) rc = cuda_fail(e, "D2D");
    }
    if (!rc) rc = batch_check_flags(b, g_stream);
    else cudaStreamSynchronize(g_stream);
    b.release();
    return rc;
}

int sipp_prove_native_batch(const uint8_t* A, const uint8_t* B, size_t n, size_t count, uint8_t* proofs) {
    int rc = ensure_init();
    if (rc) return rc;
    rc = batch_args(A, B, n, count, proofs);
    if (rc) return rc;
    const size_t np = sipp_proof_len(n);
    BatchBuffers b;
    rc = batch_alloc(b, n, count);
    if (rc) return rc;
    cudaError_t e = cudaMemcpyAsync(b.bytesA, A, n * count * 64, cudaMemcpyHostToDevice, g_stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(b.bytesB, B, n * count * 128, cudaMemcpyHostToDevice, g_stream);
    if (e != cudaSuccess) { b.release(); return cuda_fail(e, "H2D"); }
    rc = batch_prove_resident(b, n, count, g_stream);
    if (!rc) {
        e = cudaMemcpyAsync(proofs, b.proofs, count * np * 384, cudaMemcpyDeviceToHost, g_stream);
        if (e != cudaSuccess) rc = cuda_fail(e, "D2H");
    }
    if (!rc) rc = batch_check_flags(b, g_stream);
    else cudaStreamSynchronize(g_stream);
    b.release();
    return rc;
}

// sipp_prove_native_batch(_device) plus every instance's statement members (verifier_native.rs:74-75, :59-61): after the last round
// the first point of every instance is its final point, and final_Z = pairing(final_A, final_B) by bilinearity.  Nothing is copied
// to the caller before the flags passed.  in_kind / out_kind: the copies of the inputs and of every output.
static int batch_prove_statement(const void* A, const void* B, size_t n, size_t count, void* proofs, void* final_A, void* final_B, void* final_Z,
                                 cudaMemcpyKind in_kind, cudaMemcpyKind out_kind) {
    int rc = batch_args(A, B, n, count, proofs);  // the checks of sipp_prove_native_batch, before the device is touched
    if (rc) return rc;
    rc = ensure_init();
    if (rc) return rc;
    const size_t np = sipp_proof_len(n);
    BatchBuffers b;
    rc = batch_alloc(b, n, count);
    if (rc) return rc;
    uint32_t *dpair = nullptr, *dfin = nullptr;
    cudaError_t e = final_Z ? pool_alloc((void**)&dpair, count * 384) : cudaSuccess;
    if (e == cudaSuccess && (final_A || final_B)) e = pool_alloc((void**)&dfin, count * 192);
    auto run = [&]() -> int {
        if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(batch statement)");
        CK(cudaMemcpyAsync(b.bytesA, A, n * count * 64, in_kind, g_stream));
        CK(cudaMemcpyAsync(b.bytesB, B, n * count * 128, in_kind, g_stream));
        int rc2 = batch_prove_resident(b, n, count, g_stream);
        if (!rc2) rc2 = batch_finals(b, n, count, dpair, dfin, g_stream);
        if (!rc2) rc2 = batch_check_flags(b, g_stream);
        if (rc2) return rc2;
        CK(cudaMemcpyAsync(proofs, b.proofs, count * np * 384, out_kind, g_stream));
        if (final_A) CK(cudaMemcpyAsync(final_A, dfin, count * 64, out_kind, g_stream));
        if (final_B) CK(cudaMemcpyAsync(final_B, dfin + count * 16, count * 128, out_kind, g_stream));
        if (final_Z) CK(cudaMemcpyAsync(final_Z, dpair, count * 384, out_kind, g_stream));
        CK(cudaStreamSynchronize(g_stream));
        return SIPP_OK;
    };
    rc = run();
    if (rc) cudaStreamSynchronize(g_stream);
    b.release();
    pool_free(dpair);
    pool_free(dfin);
    return rc;
}

int sipp_prove_native_batch_statement(const uint8_t* A, const uint8_t* B, size_t n, size_t count, uint8_t* proofs, uint8_t* final_A,
                                      uint8_t* final_B, uint8_t* final_Z) {
    return batch_prove_statement(A, B, n, count, proofs, final_A, final_B, final_Z, cudaMemcpyHostToDevice, cudaMemcpyDeviceToHost);
}

int sipp_prove_native_batch_statement_device(const void* dA, const void* dB, size_t n, size_t count, void* d_proofs, void* d_final_A,
                                             void* d_final_B, void* d_final_Z) {
    return batch_prove_statement(dA, dB, n, count, d_proofs, d_final_A, d_final_B, d_final_Z, cudaMemcpyDeviceToDevice, cudaMemcpyDeviceToDevice);
}

// `count` independent verifications in lock-step (verifier_native.rs:14-85 per instance, batch_verify_enqueue).
// results[j] = SIPP_OK / SIPP_ERR_VERIFY / SIPP_ERR_ENCODING.
int sipp_verify_native_batch(const uint8_t* A, const uint8_t* B, size_t n, size_t count, const uint8_t* proofs, size_t proof_len, int* results,
                             uint8_t* final_A, uint8_t* final_B, uint8_t* final_Z) {
    int rc = ensure_init();
    if (rc) return rc;
    if (!results) return fail(SIPP_ERR_ARG, "null results");
    rc = batch_args(A, B, n, count, proofs);
    if (rc) return rc;
    const size_t np = sipp_proof_len(n);
    if (proof_len < np) return fail(SIPP_ERR_SHORT_PROOF, "proof.pop().unwrap() on an empty proof");  // verifier_native.rs:31,40,42
    const size_t total = n * count;
    cudaStream_t s = g_stream;
    std::vector<uint8_t> hz(count * 384), hp(count * 384);
    {
        VerifyBuffers v;
        rc = v.alloc(n, count, proof_len, true);
        if (rc) return rc;
        auto run = [&]() -> int {
            CK(cudaMemcpyAsync(v.b.bytesA, A, total * 64, cudaMemcpyHostToDevice, s));
            CK(cudaMemcpyAsync(v.b.bytesB, B, total * 128, cudaMemcpyHostToDevice, s));
            CK(cudaMemcpyAsync(v.dproofs, proofs, count * proof_len * 384, cudaMemcpyHostToDevice, s));
            int rc2 = batch_verify_enqueue(v, v.b.bytesA, v.b.bytesB, v.dproofs, n, count, proof_len, final_A || final_B, s);
            if (rc2) return rc2;
            if (final_A) CK(cudaMemcpyAsync(final_A, v.dfin, count * 64, cudaMemcpyDeviceToHost, s));
            if (final_B) CK(cudaMemcpyAsync(final_B, v.dfin + count * 16, count * 128, cudaMemcpyDeviceToHost, s));
            CK(cudaMemcpyAsync(hz.data(), v.dz, count * 384, cudaMemcpyDeviceToHost, s));
            CK(cudaMemcpyAsync(hp.data(), v.dpair, count * 384, cudaMemcpyDeviceToHost, s));
            return batch_check_flags(v.b, s);
        };
        rc = run();
        if (rc) cudaStreamSynchronize(s);
    }
    if (rc) return rc;
    for (size_t j = 0; j < count; j++) {
        // a proof with a coordinate >= p is one the reference could not have deserialised: refused on its own, like a bad A or B
        const uint8_t* pj = proofs + (j * proof_len + (proof_len - np)) * 384;
        results[j] = !fq_bytes_canonical(pj, 12 * np) ? SIPP_ERR_ENCODING
                     : memcmp(&hz[384 * j], &hp[384 * j], 384) == 0 ? SIPP_OK : SIPP_ERR_VERIFY;  // :81-84
    }
    if (final_Z) memcpy(final_Z, hz.data(), count * 384);
    return SIPP_OK;
}

// sipp_verify_native_batch on the caller's device buffers, read in place; the outcome of every instance (k_verify_outcome) goes to
// d_results and the finals only once the flags of the call were found clean.
int sipp_verify_native_batch_device(const void* dA, const void* dB, size_t n, size_t count, const void* d_proofs, size_t proof_len, int* d_results,
                                    void* d_final_A, void* d_final_B, void* d_final_Z) {
    int rc = batch_args(dA, dB, n, count, d_proofs);  // every argument check before the device is touched
    if (rc) return rc;
    if (!d_results) return fail(SIPP_ERR_ARG, "null results");
    const size_t np = sipp_proof_len(n);
    if (proof_len < np) return fail(SIPP_ERR_SHORT_PROOF, "proof.pop().unwrap() on an empty proof");  // verifier_native.rs:31,40,42
    rc = ensure_init();
    if (rc) return rc;
    cudaStream_t s = g_stream;
    std::vector<RaggedProof> pt(count);  // the elements read of proof j: its last np
    for (size_t j = 0; j < count; j++) pt[j] = RaggedProof{j * proof_len + proof_len - np, (uint32_t)np, 0};
    VerifyBuffers v;
    rc = v.alloc(n, count, proof_len, false);
    if (rc) return rc;
    RaggedProof* dpt = nullptr;
    cudaError_t e = pool_alloc((void**)&dpt, count * sizeof(RaggedProof));
    struct Release { RaggedProof* p; ~Release() { pool_free(p); } } release{dpt};
    if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(verify batch)");
    const uint32_t* proofs = (const uint32_t*)d_proofs;
    auto run = [&]() -> int {
        CK(order_after(s, cudaStreamLegacy));  // inputs just written on the legacy default stream (torch's, unless switched)
        CK(cudaMemcpyAsync(dpt, pt.data(), count * sizeof(RaggedProof), cudaMemcpyHostToDevice, s));
        int rc2 = batch_verify_enqueue(v, (const uint32_t*)dA, (const uint32_t*)dB, proofs, n, count, proof_len, d_final_A || d_final_B, s);
        if (!rc2) rc2 = batch_check_flags(v.b, s);  // synchronises
        if (rc2) return rc2;
        int le = launch_verify_outcome(proofs, dpt, count, v.dz, v.dpair, v.dfin, true, d_results, (uint32_t*)d_final_A, (uint32_t*)d_final_B,
                                       (uint32_t*)d_final_Z, s);
        if (le) return cuda_fail((cudaError_t)le, "k_verify_outcome");
        g_stats.launches++;
        CK(cudaStreamSynchronize(s));
        return SIPP_OK;
    };
    rc = run();
    if (rc) cudaStreamSynchronize(s);
    return rc;
}

// `count` independent Poseidon permutations on the device (test hook for k_transcript.cu)
int sipp_test_poseidon_device(uint64_t* states, size_t count) {
    int rc = ensure_init();
    if (rc) return rc;
    if (!states || count == 0) return fail(SIPP_ERR_ARG, "bad argument");
    uint64_t* d;
    CK(cudaMalloc(&d, count * 96));
    cudaError_t e = cudaMemcpyAsync(d, states, count * 96, cudaMemcpyHostToDevice, g_stream);
    if (e == cudaSuccess) e = (cudaError_t)launch_test_poseidon(d, count, g_stream);
    g_stats.launches++;
    if (e == cudaSuccess) e = cudaMemcpyAsync(states, d, count * 96, cudaMemcpyDeviceToHost, g_stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(g_stream);
    cudaFree(d);
    if (e != cudaSuccess) return cuda_fail(e, "sipp_test_poseidon_device");
    return SIPP_OK;
}

// device transcript of one round for `count` instances (test hook): states in/out (4 x u64 each), fq12s = count x nf x 384 B
// (nf = 2: Z_L, Z_R; nf = 3: Z, Z_L, Z_R), out: count x 64 B = x || x^-1, plans_out: count x sizeof(FoldPlan) or NULL
int sipp_test_transcript_round_device(uint64_t* states, const uint8_t* fq12s, int nf, size_t count, uint8_t* x_out, uint32_t* plans_out) {
    int rc = ensure_init();
    if (rc) return rc;
    if (!states || !fq12s || !x_out || count == 0 || (nf != 2 && nf != 3)) return fail(SIPP_ERR_ARG, "bad argument");
    uint64_t *d_st, *d_x;
    uint32_t* d_f;
    FoldPlan* d_pl;
    int* d_flags;
    CK(cudaMalloc(&d_st, count * 32));
    CK(cudaMalloc(&d_x, count * 64));
    CK(cudaMalloc(&d_f, count * nf * 384));
    CK(cudaMalloc(&d_pl, count * sizeof(FoldPlan)));
    CK(cudaMalloc(&d_flags, sizeof(int)));
    cudaMemsetAsync(d_flags, 0, sizeof(int), g_stream);
    cudaMemcpyAsync(d_st, states, count * 32, cudaMemcpyHostToDevice, g_stream);
    cudaMemcpyAsync(d_f, fq12s, count * nf * 384, cudaMemcpyHostToDevice, g_stream);
    cudaError_t e = (cudaError_t)launch_tr_round(d_st, d_f, nf, nf == 3 ? 0 : -1, nf - 2, nf - 1, g_opt_fq12_order, count, d_pl, d_x, d_flags, g_stream);
    g_stats.launches++;
    int flags = 0;
    if (e == cudaSuccess) e = cudaMemcpyAsync(states, d_st, count * 32, cudaMemcpyDeviceToHost, g_stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(x_out, d_x, count * 64, cudaMemcpyDeviceToHost, g_stream);
    if (e == cudaSuccess && plans_out) e = cudaMemcpyAsync(plans_out, d_pl, count * sizeof(FoldPlan), cudaMemcpyDeviceToHost, g_stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(&flags, d_flags, sizeof(int), cudaMemcpyDeviceToHost, g_stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(g_stream);
    cudaFree(d_st); cudaFree(d_x); cudaFree(d_f); cudaFree(d_pl); cudaFree(d_flags);
    if (e != cudaSuccess) return cuda_fail(e, "sipp_test_transcript_round_device");
    if (flags & 1) return fail(SIPP_ERR_ZERO_CHALLENGE, "challenge is zero");
    if (flags & 2) return fail(SIPP_ERR_ENCODING, "fold scalar recoding failed");
    return SIPP_OK;
}

}  // extern "C"

// sipp_b200.cu -- C ABI implementation (include/sipp_b200.h): CUDA launches + the host prover / verifier loops.
//
// Host control flow mirrors /root/reference/src/prover_native.rs:26-80 and verifier_native.rs:14-85 line by line
// (cited inline); all group / field arithmetic runs in the kernels of kernels.cuh.  There is no CPU arithmetic
// fallback: every compute entry point returns SIPP_ERR_CUDA when no device is usable.
#include <cuda_runtime.h>
#include <stdio.h>
#include <string.h>

#include <chrono>
#include <string>
#include <thread>
#include <vector>

#include "glv_core.h"
#include "host_state.h"

using namespace sipp;

namespace sipp_host {

thread_local std::string g_err;
int g_device = -1;
cudaStream_t g_stream = nullptr;
int g_opt_fe_norm = 0, g_opt_fq12_order = 0, g_opt_profile = 0, g_opt_pipeline = 1;
int g_opt_fe_engine = 1;
int g_opt_wide_fold_max = 256;
int g_opt_wide_accum_max = 1536;
int g_opt_wide_max = 8192;  // pairs per launch up to which the 16-lanes-per-pair line kernel is used (latency-bound rounds)
int g_sm_count = 148;
int g_opt_fold_straus = 1;     // throughput folds (batched instances, large rounds): 1 = one thread per element, shared doublings
int g_opt_batch_streams = 0;   // batched instances: sub-batches on their own streams (0 = choose by batch size)
int g_opt_batch_qlines = 1;    // batched instances: Q-only line coefficients computed once for Z and the first Z_L / Z_R
int g_opt_batch_kpg_max = 32;  // batched instances: pairs of one product that share an accumulator group, at most
int g_opt_matrix_n = 32;       // pairing matrix of single points (k_mat.cu) once at most this many points are left; 0 = off
int g_opt_matrix_first = 1;     // the first matrix is built from the inputs, under the host's absorb chain; 10..24: log2 of its Miller-loop budget
int g_opt_matrix_block_n = 256, g_opt_matrix_block_r = 8;  // look-ahead stages: from at most this many points, that many blocks
int g_opt_validate = 1;        // every prove / verify entry point checks its points: on the curve, B_i in the order-r subgroup
int g_opt_product_chunk = 0;    // batched independent products (products.cu): pairs per line-table chunk, at most; 0 = by the budget

struct TimedSpan {
    cudaEvent_t a, b;
    int kind;  // 0 miller, 1 reduce_fe, 2 fold, 3 other
};
std::vector<TimedSpan> g_spans;
sipp_stats g_stats;

int fail(int code, const char* what) {
    g_err = what;
    return code;
}
int cuda_fail(cudaError_t e, const char* what) {
    g_err = std::string(what) + ": " + cudaGetErrorString(e);
    return SIPP_ERR_CUDA;
}
int ensure_init() {
    if (g_device >= 0) return SIPP_OK;
    return sipp_init(0);
}

int span_begin(int kind, cudaStream_t s) {
    if (!g_opt_profile) return -1;
    TimedSpan t;
    t.kind = kind;
    cudaEventCreate(&t.a);
    cudaEventCreate(&t.b);
    cudaEventRecord(t.a, s);
    g_spans.push_back(t);
    return (int)g_spans.size() - 1;
}
void span_end(int idx, cudaStream_t s) {
    if (idx >= 0) cudaEventRecord(g_spans[idx].b, s);
}

void collect_spans() {
    for (auto& t : g_spans) {
        cudaEventSynchronize(t.b);
        float ms = 0;
        cudaEventElapsedTime(&ms, t.a, t.b);
        if (t.kind == 0) g_stats.miller_ms += ms;
        else if (t.kind == 1) g_stats.reduce_fe_ms += ms;
        else if (t.kind == 2) g_stats.fold_ms += ms;
        else g_stats.other_ms += ms;
        cudaEventDestroy(t.a);
        cudaEventDestroy(t.b);
    }
    g_spans.clear();
}

double AbsorbJob::join() {
    if (!th.joinable()) return 0.0;
    auto t0 = std::chrono::steady_clock::now();
    th.join();
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
}

size_t log2_exact(size_t n) {
    size_t r = 0;
    while (n > 1) { n >>= 1; r++; }
    return r;
}
bool is_pow2(size_t n) { return n && !(n & (n - 1)); }

Scalar256 scalar_from_bytes(const uint8_t* b) {
    Scalar256 s;
    memcpy(s.w, b, 32);
    return s;
}

// The scalars of one fold (prover_native.rs:58-69, verifier_native.rs:46-61): x and x_inv canonical (< r), x != 0, x x_inv = 1 (mod r).
// The kernels only see the recodings, which would reduce a scalar >= r silently; a wrong inverse would fold B by whatever it is given
// and, on the pairing-matrix route, give other Z_L / Z_R than the point route.  Host only: one Fr product, no device work.
int check_fold_scalars(const uint8_t* x, const uint8_t* x_inv) {
    const uint64_t R[4] = {0x43e1f593f0000001ull, 0x2833e84879b97091ull, 0xb85045b68181585dull, 0x30644e72e131a029ull};
    const uint64_t R2[4] = {0x1bb8e645ae216da7ull, 0x53fe3ab1e35c59e3ull, 0x8c49833d53bb8085ull, 0x0216d0b17f4e44a5ull};  // 2^512 mod r
    uint64_t a[4], b[4], t[4];
    memcpy(a, x, 32);
    memcpy(b, x_inv, 32);
    if (glv::fr_geq(a, R) || glv::fr_geq(b, R)) return fail(SIPP_ERR_ENCODING, "fold scalar out of range (must be < r)");
    if (!(a[0] | a[1] | a[2] | a[3])) return fail(SIPP_ERR_ZERO_CHALLENGE, "challenge is zero: x.inverse().unwrap() panics in the reference");
    glv::fr_mont_mul(t, a, b);   // x x_inv / 2^256
    glv::fr_mont_mul(t, t, R2);  // x x_inv
    if (t[0] != 1 || (t[1] | t[2] | t[3])) return fail(SIPP_ERR_ENCODING, "x_inv is not the inverse of x");
    return SIPP_OK;
}

// Device memory pool: contexts and staging buffers are created per prove call; cudaMalloc / cudaFree cost hundreds of
// microseconds each and cudaFree synchronises the device, so freed blocks are kept and reused (grow-only, released in
// sipp_shutdown).  One host thread per process by contract, so no locking.
struct PoolBlock {
    void* ptr;
    size_t size;
    bool used;
};
std::vector<PoolBlock> g_pool;
cudaError_t pool_alloc(void** out, size_t bytes) {
    if (bytes == 0) bytes = 16;
    int best = -1;
    for (size_t i = 0; i < g_pool.size(); i++) {
        const PoolBlock& b = g_pool[i];
        if (!b.used && b.size >= bytes && b.size <= 2 * bytes && (best < 0 || b.size < g_pool[best].size)) best = (int)i;
    }
    if (best >= 0) {
        g_pool[best].used = true;
        *out = g_pool[best].ptr;
        return cudaSuccess;
    }
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e != cudaSuccess) return e;
    g_pool.push_back({p, bytes, true});
    *out = p;
    return cudaSuccess;
}
void pool_free(void* p) {
    if (!p) return;
    for (auto& b : g_pool)
        if (b.ptr == p) { b.used = false; return; }
    cudaFree(p);  // not from the pool
}
void pool_release_all() {
    for (auto& b : g_pool) cudaFree(b.ptr);
    g_pool.clear();
}

// device scratch shared by all contexts of this process (one host thread per process by contract)
struct Scratch {
    uint32_t* partials = nullptr;  // [blocks][2][96]
    size_t partial_blocks = 0;
    uint32_t* out = nullptr;       // 4 x 96 words device result
    uint8_t* h_out = nullptr;      // pinned mirror
    int* flag = nullptr;
    int* vflag = nullptr;          // result of a deferred point validation (sipp_prove_native / sipp_verify_native)
    uint32_t* lines = nullptr;     // split pipeline: [nprod][mc][91][80 words]
    size_t lines_bytes = 0;
} g_scr;

int scratch_reserve(size_t blocks) {
    if (!g_scr.out) {
        CK(cudaMalloc(&g_scr.out, 4 * 96 * sizeof(uint32_t)));
        CK(cudaMallocHost(&g_scr.h_out, 4 * 384));
        CK(cudaMalloc(&g_scr.flag, sizeof(int)));
        CK(cudaMalloc(&g_scr.vflag, sizeof(int)));
    }
    if (blocks > g_scr.partial_blocks) {
        if (g_scr.partials) CK(cudaFree(g_scr.partials));
        size_t cap = blocks < 1024 ? 1024 : blocks;
        CK(cudaMalloc(&g_scr.partials, cap * 2 * 96 * sizeof(uint32_t)));
        g_scr.partial_blocks = cap;
    }
    return SIPP_OK;
}

int lines_reserve(size_t bytes) {
    if (bytes > g_scr.lines_bytes) {
        if (g_scr.lines) CK(cudaFree(g_scr.lines));
        g_scr.lines = nullptr;
        g_scr.lines_bytes = 0;
        CK(cudaMalloc(&g_scr.lines, bytes));
        g_scr.lines_bytes = bytes;
    }
    return SIPP_OK;
}

uint32_t* lines_buffer() { return g_scr.lines; }

cudaError_t order_after(cudaStream_t later, cudaStream_t earlier) {
    cudaEvent_t ev;
    cudaError_t e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
    if (e != cudaSuccess) return e;
    e = cudaEventRecord(ev, earlier);
    if (e == cudaSuccess) e = cudaStreamWaitEvent(later, ev, 0);
    cudaEventDestroy(ev);
    return e;
}


}  // namespace sipp_host
using namespace sipp_host;

namespace {

// decode boundary bytes already on the device (d_bytes) into Montgomery limbs (d_out); n_fq field elements
int launch_decode(const uint32_t* d_bytes, uint32_t* d_out, size_t n_fq, cudaStream_t s, bool check) {
    if (check) CK(cudaMemsetAsync(g_scr.flag, 0, sizeof(int), s));
    Span sp(3, s);
    int e = launch_codec_decode(d_bytes, d_out, n_fq, check ? g_scr.flag : nullptr, s);
    if (e) return cuda_fail((cudaError_t)e, "k_codec_decode");
    g_stats.launches++;
    return SIPP_OK;
}

// launches the Miller kernel for `nprod` products of m pairs each; returns the number of partial sets (blocks)
int launch_miller(const sipp_ctx* c, int nprod, const MillerJob& job, uint32_t* d_partials, size_t* blocks_out, cudaStream_t s) {
    size_t blocks = (job.m + SIPP_MILLER_BLOCK - 1) / SIPP_MILLER_BLOCK;
    {
        Span sp(0, s);
        int e = launch_miller_block(c->dA, c->dB, job, nprod, d_partials, s);
        if (e) return cuda_fail((cudaError_t)e, "k_miller_block");
    }
    g_stats.launches++;
    g_stats.miller_launches++;
    g_stats.miller_pairs += job.m * (size_t)nprod;
    *blocks_out = blocks;
    return SIPP_OK;
}

int launch_reduce(const uint32_t* d_partials, int count, int nprod, uint32_t* d_out, bool final_exp, cudaStream_t s) {
    Span sp(1, s);
    int e = !g_opt_pipeline ? launch_reduce_fe(d_partials, count, nprod, d_out, final_exp ? 1 : 0, g_opt_fe_norm, s)
            : g_opt_fe_engine ? launch_reduce_fe_eng(d_partials, count, nprod, d_out, final_exp ? 1 : 0, g_opt_fe_norm, s)
                              : launch_reduce_fe_coop(d_partials, count, nprod, d_out, final_exp ? 1 : 0, g_opt_fe_norm, s);
    if (e) return cuda_fail((cudaError_t)e, "k_reduce_fe");
    g_stats.launches++;
    return SIPP_OK;
}

// products for the current round: which = 0 -> Z over all n pairs; which = 1 -> Z_L, Z_R over the crossed halves
int ctx_products_to_device(sipp_ctx* c, int which, size_t* blocks_out, int* nprod_out, cudaStream_t s) {
    MillerJob job;
    int nprod;
    if (which == 0) {
        nprod = 1;
        job.a_off[0] = 0; job.b_off[0] = 0; job.a_off[1] = 0; job.b_off[1] = 0;
        job.m = c->n;
    } else {
        if (c->n < 2) return fail(SIPP_ERR_ARG, "cross products need n >= 2");
        size_t h = c->n / 2;
        nprod = 2;
        job.a_off[0] = h; job.b_off[0] = 0;  // Z_L = inner_product(A2, B1)   prover_native.rs:48
        job.a_off[1] = 0; job.b_off[1] = h;  // Z_R = inner_product(A1, B2)   prover_native.rs:49
        job.m = h;
    }
    *nprod_out = nprod;
    if (!g_opt_pipeline) {
        size_t blocks = (job.m + SIPP_MILLER_BLOCK - 1) / SIPP_MILLER_BLOCK;
        int rc = scratch_reserve(blocks);
        if (rc) return rc;
        return launch_miller(c, nprod, job, g_scr.partials, blocks_out, s);
    }
    // split pipeline: L (lines -> HBM) then A (6-lane cooperative accumulation), in chunks that bound the line buffer
    const size_t per_pair = lines_bytes_per_pair();
    const size_t cap_bytes = (size_t)6 << 30;
    size_t mc = job.m;
    if (mc * (size_t)nprod * per_pair > cap_bytes) mc = cap_bytes / ((size_t)nprod * per_pair);
    // accumulation: 6-lane groups (k_accum, 20 per block) or, for the small launches of the latency-bound rounds, one
    // 32-lane machine per group (k_accum_eng, 4 per block); kpg pairs share one accumulator (and its squarings)
    const bool eng = mc * (size_t)nprod <= (size_t)g_opt_wide_accum_max;
    const size_t groups_target = eng ? (size_t)g_sm_count * 8 : (size_t)g_sm_count * 2 * 20;
    int kpg = (int)(((eng ? mc * (size_t)nprod : mc) + groups_target - 1) / groups_target);
    if (kpg < 1) kpg = 1;
    auto blocks_of = [&](size_t cur) { return (size_t)(eng ? accum_eng_blocks(cur, kpg) : accum_blocks(cur, kpg)); };
    size_t total_blocks = 0;
    for (size_t c0 = 0; c0 < job.m; c0 += mc) {
        size_t cur = job.m - c0 < mc ? job.m - c0 : mc;
        total_blocks += blocks_of(cur);
    }
    int rc = scratch_reserve(total_blocks);
    if (rc) return rc;
    rc = lines_reserve(mc * (size_t)nprod * per_pair);
    if (rc) return rc;
    size_t block_off = 0;
    for (size_t c0 = 0; c0 < job.m; c0 += mc) {
        size_t cur = job.m - c0 < mc ? job.m - c0 : mc;
        Span sp(0, s);
        const bool wide = cur * (size_t)nprod <= (size_t)g_opt_wide_max;
        int e = wide ? launch_lines_wide(c->dA, c->dB, job, nprod, c0, cur, g_scr.lines, s) : launch_lines(c->dA, c->dB, job, nprod, c0, cur, g_scr.lines, s);
        if (e) return cuda_fail((cudaError_t)e, "k_lines");
        e = eng ? launch_accum_eng(g_scr.lines, cur, nprod, kpg, g_scr.partials, (int)block_off, s)
                : launch_accum(g_scr.lines, cur, nprod, kpg, g_scr.partials, (int)block_off, s);
        if (e) return cuda_fail((cudaError_t)e, "k_accum");
        block_off += blocks_of(cur);
        g_stats.launches += 2;
        g_stats.miller_launches++;
    }
    g_stats.miller_pairs += job.m * (size_t)nprod;
    *blocks_out = total_blocks;
    return SIPP_OK;
}

int ctx_products(sipp_ctx* c, int which, uint8_t* out0, uint8_t* out1) {
    size_t blocks;
    int nprod;
    int rc = ctx_products_to_device(c, which, &blocks, &nprod, g_stream);
    if (rc) return rc;
    rc = launch_reduce(g_scr.partials, (int)blocks, nprod, g_scr.out, true, g_stream);
    if (rc) return rc;
    CK(cudaMemcpyAsync(g_scr.h_out, g_scr.out, (size_t)nprod * 384, cudaMemcpyDeviceToHost, g_stream));
    CK(cudaStreamSynchronize(g_stream));
    memcpy(out0, g_scr.h_out, 384);
    if (nprod == 2) memcpy(out1, g_scr.h_out + 384, 384);
    return SIPP_OK;
}

}  // namespace

namespace sipp_host {
// ---- pairing-matrix stages (k_mat.cu).  The rounds of prover_native.rs:45-75 are a serial chain fold -> Miller loops -> final
// exponentiation -> hash; bilinearity cuts it.  Split the n points left into nr blocks of m = n / nr ("virtual points") and let
//     E[i][j] = <A_block_i, B_block_j> = prod_{t<m} e(A[i m + t], B[j m + t])        (all nr^2 block products, ONE launch set).
// Then Z_L = prod_{i<nr/2} E[i + nr/2][i], Z_R = prod E[i][i + nr/2] (:48-49), and the fold of the points (:60-69) carries over to
// the matrix: E'[i][j] = E[i][j] E[i+h][j+h] E[i+h][j]^x E[i][j+h]^(1/x) -- one short kernel (k_mat_fold) -- for log2(nr) rounds.
//   m == 1 (n <= SIPP_OPT_MATRIX_TAIL): the tail of the proof; the points are never folded again.
//   m > 1  (n <= SIPP_OPT_MATRIX_BLOCK_N): a look-ahead stage of log2(nr) rounds; the points are folded with every challenge on a
//          side stream, off the critical path, and the next stage starts from them.
// Every Z_L, Z_R is the same field element as on the point-fold route, bit for bit.
cudaStream_t g_fold_stream = nullptr;
FoldPlan* g_fold_plan_dev = nullptr;  // device copy of the plan for k_fold_straus (released in sipp_shutdown)
int g_live_ctx = 0;                   // contexts alive (a device switch is refused while any exists)

// Stage sizes (measured on B200, tools/tail_ab.py, profiles/r02_v7_stage_ab.txt).  A matrix of single points pays from 32 points
// down (1,024 Miller loops + final exponentiations in one latency); a look-ahead stage takes n / 16 blocks, at most
// SIPP_OPT_MATRIX_BLOCK_R (it ends at 16 or 32 points, where the matrix of single points takes over); the first stage takes n / 32 blocks, between 8 and 32, as long as the launch stays under 2^17 loops
// (more blocks than that and the matrix no longer fits under the absorb chain of a small proof: n = 512 with 32 blocks lost 1 ms).
size_t mat_stage(size_t n) {
    if (!g_opt_pipeline || !g_opt_fe_engine || n < 2) return 0;
    if (n <= (size_t)g_opt_matrix_n) return n;
    if (g_opt_matrix_n < 2 || n > (size_t)g_opt_matrix_block_n) return 0;
    size_t nr = n / 16;
    if (nr > (size_t)g_opt_matrix_block_r) nr = (size_t)g_opt_matrix_block_r;
    while (nr >= 4 && n / nr < 2) nr >>= 1;
    return nr >= 4 ? nr : 0;
}

// The FIRST stage of a proof starts from the inputs themselves, before any challenge exists: it runs in the shadow of the host's
// 8n-permutation absorb chain, gives Z as the product of its diagonal, and the first log2(nr) rounds cost one matrix fold each.
// Miller loops the first stage may spend.  It has to finish inside the host's absorb of the same inputs: 8 n permutations of 0.67 us
// against ~6 M loops/s plus ~2.5 ms of fixed work (validation, line coefficients, final exponentiations), i.e. about 32 n - 15,000
// loops.  Measured on the box (tools/first_ab.py, profiles/r02_v8_first_stage_ab.txt): best are n / 128 blocks from n = 2^9 (4 blocks)
// to 2^12 (32 blocks: slightly over, but it saves a round), 8 blocks at 2^8, 32 n loops above; the absolute cap bounds the line
// table (29 KB per loop).
size_t mat_first_budget(size_t n) {
    if (g_opt_matrix_first >= 10) return (size_t)1 << g_opt_matrix_first;
    const size_t by_n = n <= 256 ? 16 * n : n < 4096 ? n * (n / 128) : 32 * n, cap = (size_t)1 << SIPP_FIRST_STAGE_LOG2_LOOPS;
    return by_n < cap ? by_n : cap;
}
size_t mat_stage_first(size_t n) {
    if (!g_opt_matrix_first || !g_opt_pipeline || !g_opt_fe_engine || n < 2 || g_opt_matrix_n < 2) return 0;
    if (n <= (size_t)g_opt_matrix_n) return n;               // the whole proof on the matrix of its inputs
    size_t nr = n / 32;
    if (nr < 8) nr = 8;
    if (nr > 32) nr = 32;
    while (nr > 1 && nr * n > mat_first_budget(n)) nr >>= 1;  // n nr Miller loops
    while (nr >= 4 && n / nr < 2) nr >>= 1;
    return nr >= 4 ? nr : 0;
}

int mat_build(sipp_ctx* c, MatTail& mt, size_t nr) { return mat_build_ex(c, mt, nr, nullptr); }

// raw_out != NULL (a rank of the sharded prover): only this shard's UN-exponentiated entry products are computed and written there
// (nr^2 x 96 words, register-shaped) -- they are all-gathered and rank 0 finishes with mat_adopt; `mt` is not touched
int mat_build_ex(sipp_ctx* c, MatTail& mt, size_t nr, uint32_t* raw_out) {
    const size_t n = c->n, m = n / nr, P = nr * nr, pairs = P * m;
    // small launches: the lane engines (latency); large ones (a first stage): line coefficients of every B point once + the
    // throughput accumulation kernel
    const bool big = m > 1 && pairs > 8192;
    int kpg = 1;
    if (big) {
        const size_t by_block = (m + 19) / 20, by_fill = (pairs + 11839) / 11840;
        kpg = (int)(by_block < by_fill ? by_block : by_fill);
        if (kpg < 1) kpg = 1;
    }
    const size_t blocks = big ? (size_t)accum_blocks(m, kpg) : (size_t)accum_eng_blocks(m, 1);
    uint32_t *aexp = nullptr, *bexp = nullptr, *mil = nullptr, *ql = nullptr, *prod = nullptr;
    int rc = scratch_reserve(m == 1 ? nr : (blocks * P + 1) / 2);
    if (!rc) rc = lines_reserve(pairs * lines_bytes_per_pair());
    if (rc) return rc;
    cudaError_t e = cudaSuccess;
    if (!raw_out) {
        e = pool_alloc((void**)&mt.E[0], P * 384);
        if (e == cudaSuccess) e = pool_alloc((void**)&mt.E[1], (P / 4) * 384);
    }
    if (e == cudaSuccess && !big) e = pool_alloc((void**)&aexp, pairs * 64);
    if (e == cudaSuccess && !big) e = pool_alloc((void**)&bexp, pairs * 128);
    if (e == cudaSuccess && big) e = pool_alloc((void**)&ql, n * qlines_bytes_per_point());
    if (e == cudaSuccess && m == 1 && !raw_out) e = pool_alloc((void**)&mil, P * 384);
    if (m == 1 && raw_out) mil = raw_out;
    int le = 0;
    if (e == cudaSuccess) {
        {
            Span sp(0, g_stream);
            if (big) {
                le = launch_qlines_batch(c->dB, n, ql, g_stream);
                if (!le) le = launch_eval_lines_mat(c->dA, c->dB, nr, m, ql, g_scr.lines, g_stream);
                // the expanded launch is laid out [entry][pair of the block]: an entry is one "product" of m pairs
                if (!le) le = launch_accum(g_scr.lines, m, (int)P, kpg, g_scr.partials, 0, g_stream);
            } else {
                MillerJob job;
                job.a_off[0] = job.b_off[0] = job.a_off[1] = job.b_off[1] = 0;
                job.m = pairs;
                le = launch_mat_gather(c->dA, c->dB, nr, m, aexp, bexp, g_stream);
                if (!le)
                    le = pairs <= (size_t)g_opt_wide_max ? launch_lines_wide(aexp, bexp, job, 1, 0, pairs, g_scr.lines, g_stream)
                                                         : launch_lines(aexp, bexp, job, 1, 0, pairs, g_scr.lines, g_stream);
                if (!le) le = m == 1 ? launch_accum_eng_each(g_scr.lines, P, mil, g_stream) : launch_accum_eng(g_scr.lines, m, (int)P, 1, g_scr.partials, 0, g_stream);
            }
        }
        if (!le && raw_out) {
            Span sp(1, g_stream);  // product of the entry's partials, no exponentiation
            if (m > 1) le = launch_reduce_fe_eng(g_scr.partials, (int)blocks, (int)P, raw_out, 0, g_opt_fe_norm, g_stream);
        } else if (!le) {
            // one final exponentiation per entry on k_mat_fe (4 machines per block, 3 blocks per SM: 1,024 entries in 1.1 ms; the
            // reduction kernel's blocks are register-bound at 2 per SM and took 3.7 ms); entries accumulated by several blocks are
            // multiplied together first (raw product, in place of the first block's partials)
            Span sp(1, g_stream);
            const uint32_t* src = m == 1 ? mil : g_scr.partials;
            if (m > 1 && blocks > 1) {
                if (pool_alloc((void**)&prod, P * 384) != cudaSuccess) le = (int)cudaErrorMemoryAllocation;
                if (!le) le = launch_reduce_fe_eng(g_scr.partials, (int)blocks, (int)P, prod, 0, g_opt_fe_norm, g_stream);
                src = prod;
                g_stats.launches++;
            }
            if (!le) le = launch_mat_fe(src, P, mt.E[0], g_opt_fe_norm, g_stream);
        }
        g_stats.launches += 4;
        g_stats.miller_launches++;
        g_stats.miller_pairs += pairs;  // Miller loops these launches compute
    }
    // the staging blocks are only reused by later work on the same stream
    pool_free(aexp);
    pool_free(bexp);
    if (mil != raw_out) pool_free(mil);
    pool_free(ql);
    pool_free(prod);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(pairing matrix)");
    if (le) return cuda_fail((cudaError_t)le, "pairing matrix");
    if (raw_out) return SIPP_OK;
    mt.n = nr;
    mt.m = m;
    mt.fold_points = m > 1;
    mt.cur = 0;
    mt.folds = 0;
    return SIPP_OK;
}

// rank 0 of the sharded prover: the matrix from the gathered entry products of all ranks (layout [rank][nr^2][96 words]): product over
// the ranks + one final exponentiation per entry.  The points of this rank's shard keep being folded with every challenge.
int mat_adopt(MatTail& mt, const uint32_t* gathered, int ranks, size_t nr) {
    const size_t P = nr * nr;
    int rc = scratch_reserve(nr);
    if (rc) return rc;
    cudaError_t e = pool_alloc((void**)&mt.E[0], P * 384);
    if (e == cudaSuccess) e = pool_alloc((void**)&mt.E[1], (P / 4) * 384);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(pairing matrix)");
    {
        Span sp(1, g_stream);
        int le = launch_reduce_fe_eng(gathered, ranks, (int)P, mt.E[0], 3, g_opt_fe_norm, g_stream);
        if (le) return cuda_fail((cudaError_t)le, "pairing matrix (gathered)");
    }
    g_stats.launches++;
    mt.n = nr;
    mt.m = 2;  // blocks of several points (spread over the ranks)
    mt.fold_points = true;
    mt.cur = 0;
    mt.folds = 0;
    return SIPP_OK;
}

// Z = prod E[i][i]   (prover_native.rs:29) from a matrix built over the inputs
int mat_diag_product(MatTail& mt, uint8_t* z) {
    {
        Span sp(1, g_stream);
        int le = launch_mat_diag(mt.E[mt.cur], mt.n, 1, g_scr.partials, g_stream);
        if (!le) le = launch_reduce_fe_eng(g_scr.partials, (int)mt.n, 1, g_scr.out, 2, g_opt_fe_norm, g_stream);
        if (le) return cuda_fail((cudaError_t)le, "matrix diagonal");
    }
    g_stats.launches += 2;
    CK(cudaMemcpyAsync(g_scr.h_out, g_scr.out, 384, cudaMemcpyDeviceToHost, g_stream));
    CK(cudaStreamSynchronize(g_stream));
    memcpy(z, g_scr.h_out, 384);
    return SIPP_OK;
}

// Z_L = prod E[i+h][i], Z_R = prod E[i][i+h]   (prover_native.rs:48-49)
int mat_products(MatTail& mt, uint8_t* zl, uint8_t* zr) {
    const size_t h = mt.n / 2;
    {
        Span sp(1, g_stream);
        int le = launch_mat_diag(mt.E[mt.cur], mt.n, 0, g_scr.partials, g_stream);
        if (!le) le = launch_reduce_fe_eng(g_scr.partials, (int)h, 2, g_scr.out, 2, g_opt_fe_norm, g_stream);
        if (le) return cuda_fail((cudaError_t)le, "matrix products");
    }
    g_stats.launches += 2;
    CK(cudaMemcpyAsync(g_scr.h_out, g_scr.out, 2 * 384, cudaMemcpyDeviceToHost, g_stream));
    CK(cudaStreamSynchronize(g_stream));
    memcpy(zl, g_scr.h_out, 384);
    memcpy(zr, g_scr.h_out + 384, 384);
    return SIPP_OK;
}

// E'[i][j] = E[i][j] E[i+h][j+h] E[i+h][j]^x E[i][j+h]^(x^-1)   (prover_native.rs:60-69 in GT); c->n halves.  A look-ahead stage
// (m > 1) also folds the points themselves, on the side stream; when the matrix is used up the library stream waits for them.
int mat_fold(sipp_ctx* c, MatTail& mt, const uint8_t x[32], const uint8_t xinv[32]) {
    if (mt.n > 2) {  // the 1 x 1 matrix after the last round of a stage is never read
        GtPlan plan;
        if (gt_plan_build(x, xinv, &plan)) return fail(SIPP_ERR_ENCODING, "fold scalar out of range (must be < r)");
        Span sp(2, g_stream);
        int le = launch_mat_fold(mt.E[mt.cur], mt.n, mt.E[mt.cur ^ 1], plan, g_stream);
        if (le) return cuda_fail((cudaError_t)le, "k_mat_fold");
        g_stats.launches++;
        mt.cur ^= 1;
    }
    const size_t h = c->n / 2;
    if (mt.fold_points) {
        FoldPlan fp;
        if (fold_plan_build(x, xinv, &fp)) return fail(SIPP_ERR_ENCODING, "fold scalar out of range (must be < r)");
        if (!g_fold_stream) CK(cudaStreamCreateWithFlags(&g_fold_stream, cudaStreamNonBlocking));
        if (mt.folds++ == 0) CK(order_after(g_fold_stream, g_stream));  // the gather of mat_build has read the points
        Span sp(2, g_fold_stream);
        int le = h <= (size_t)g_opt_wide_fold_max ? launch_fold_wide(c->dA, c->dB, h, fp, g_fold_stream) : launch_fold(c->dA, c->dB, h, fp, g_fold_stream);
        if (le) return cuda_fail((cudaError_t)le, "k_fold (look-ahead stage)");
        g_stats.launches++;
    }
    if (!mt.fold_points) c->stale = true;  // the tail: the points are not folded any more
    g_stats.fold_points += h;
    c->n = h;
    mt.n /= 2;
    if (mt.n == 1) {  // stage over
        if (mt.fold_points) CK(order_after(g_stream, g_fold_stream));
        mt.reset();
    }
    return SIPP_OK;
}

int ctx_alloc(size_t n, sipp_ctx** out) {
    sipp_ctx* c = new sipp_ctx();
    g_live_ctx++;
    c->n = c->cap = n;
    cudaError_t e = pool_alloc((void**)&c->dA, n * 16 * sizeof(uint32_t));
    if (e == cudaSuccess) e = pool_alloc((void**)&c->dB, n * 32 * sizeof(uint32_t));
    if (e != cudaSuccess) {
        pool_free(c->dA);
        delete c;
        g_live_ctx--;
        return cuda_fail(e, "cudaMalloc(ctx)");
    }
    *out = c;
    return SIPP_OK;
}
}  // namespace sipp_host

extern "C" {

const char* sipp_last_error(void) { return g_err.c_str(); }

int sipp_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

int sipp_init(int device) {
    int n = sipp_device_count();
    if (n <= 0) return fail(SIPP_ERR_CUDA, "no CUDA device: libsipp_b200 has no CPU fallback");
    if (device < 0 || device >= n) return fail(SIPP_ERR_ARG, "device index out of range");
    if (g_device >= 0 && g_device != device) {
        // a device switch: everything the library holds belongs to the old device.  Live contexts would dangle (their points are
        // pool blocks), so the switch is refused while any exists; otherwise the old device is shut down completely.
        if (g_live_ctx > 0) return fail(SIPP_ERR_ARG, "sipp_init: contexts of the current device are still alive (destroy them before switching devices)");
        CK(cudaSetDevice(g_device));
        sipp_shutdown();
    }
    CK(cudaSetDevice(device));
    if (!g_stream) CK(cudaStreamCreateWithFlags(&g_stream, cudaStreamNonBlocking));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    g_sm_count = prop.multiProcessorCount;
    g_device = device;
    return SIPP_OK;
}

int sipp_shutdown(void) {
    if (g_device < 0) return SIPP_OK;
    collect_spans();
    sipp_comm_destroy();
    if (g_scr.partials) cudaFree(g_scr.partials);
    if (g_scr.out) cudaFree(g_scr.out);
    if (g_scr.h_out) cudaFreeHost(g_scr.h_out);
    if (g_scr.flag) cudaFree(g_scr.flag);
    if (g_scr.vflag) cudaFree(g_scr.vflag);
    if (g_scr.lines) cudaFree(g_scr.lines);
    g_scr = Scratch();
    pool_release_all();
    batch_release_streams();
    if (g_fold_plan_dev) cudaFree(g_fold_plan_dev);
    g_fold_plan_dev = nullptr;
    if (g_stream) cudaStreamDestroy(g_stream);
    g_stream = nullptr;
    if (g_fold_stream) cudaStreamDestroy(g_fold_stream);
    g_fold_stream = nullptr;
    g_device = -1;
    return SIPP_OK;
}

int sipp_set_option(int option, int value) {
    switch (option) {
        case SIPP_OPT_FE_NORMALISATION: g_opt_fe_norm = value ? 1 : 0; return SIPP_OK;
        case SIPP_OPT_FQ12_ORDER: g_opt_fq12_order = value ? 1 : 0; return SIPP_OK;
        case SIPP_OPT_PROFILE: g_opt_profile = value ? 1 : 0; return SIPP_OK;
        case SIPP_OPT_PIPELINE: g_opt_pipeline = value ? 1 : 0; return SIPP_OK;
        case SIPP_OPT_WIDE_LINES_MAX: g_opt_wide_max = value < 0 ? 0 : value; return SIPP_OK;
        case SIPP_OPT_FE_ENGINE: g_opt_fe_engine = value ? 1 : 0; return SIPP_OK;
        case SIPP_OPT_WIDE_FOLD_MAX: g_opt_wide_fold_max = value < 0 ? 0 : value; return SIPP_OK;
        case SIPP_OPT_WIDE_ACCUM_MAX: g_opt_wide_accum_max = value < 0 ? 0 : value; return SIPP_OK;
        case SIPP_OPT_BATCH_KPG_MAX: g_opt_batch_kpg_max = value < 1 ? 1 : value; return SIPP_OK;
        case SIPP_OPT_FOLD_STRAUS: g_opt_fold_straus = value ? 1 : 0; return SIPP_OK;
        case SIPP_OPT_BATCH_STREAMS: g_opt_batch_streams = value < 0 ? 0 : value; return SIPP_OK;
        case SIPP_OPT_BATCH_QLINES: g_opt_batch_qlines = value ? 1 : 0; return SIPP_OK;
        case SIPP_OPT_VALIDATE_POINTS: g_opt_validate = value ? 1 : 0; return SIPP_OK;
        case SIPP_OPT_PRODUCT_CHUNK_PAIRS: g_opt_product_chunk = value < 0 ? 0 : value; return SIPP_OK;
        case SIPP_OPT_MATRIX_TAIL:
            if (value < 0 || value > 64 || (value & (value - 1))) return fail(SIPP_ERR_ARG, "SIPP_OPT_MATRIX_TAIL: 0 or a power of two <= 64");
            g_opt_matrix_n = value;
            return SIPP_OK;
        case SIPP_OPT_MATRIX_FIRST: g_opt_matrix_first = (value >= 10 && value <= 24) ? value : (value ? 1 : 0); return SIPP_OK;
        case SIPP_OPT_MATRIX_BLOCK_N: g_opt_matrix_block_n = value < 0 ? 0 : (value > 4096 ? 4096 : value); return SIPP_OK;
        case SIPP_OPT_MATRIX_BLOCK_R:
            if (value < 4 || value > 32 || (value & (value - 1))) return fail(SIPP_ERR_ARG, "SIPP_OPT_MATRIX_BLOCK_R: 4, 8, 16 or 32");
            g_opt_matrix_block_r = value;
            return SIPP_OK;
        default: return fail(SIPP_ERR_ARG, "unknown option");
    }
}
// host-side stage policy, no device needed: blocks of the first stage (which >= 0: 0 = first stage, 1 = a later stage) for n points
long sipp_test_stage_blocks(int which, size_t n) { return (long)(which == 0 ? mat_stage_first(n) : mat_stage(n)); }
int sipp_get_option(int option) {
    switch (option) {
        case SIPP_OPT_FE_NORMALISATION: return g_opt_fe_norm;
        case SIPP_OPT_FQ12_ORDER: return g_opt_fq12_order;
        case SIPP_OPT_PROFILE: return g_opt_profile;
        case SIPP_OPT_PIPELINE: return g_opt_pipeline;
        case SIPP_OPT_WIDE_LINES_MAX: return g_opt_wide_max;
        case SIPP_OPT_FE_ENGINE: return g_opt_fe_engine;
        case SIPP_OPT_WIDE_FOLD_MAX: return g_opt_wide_fold_max;
        case SIPP_OPT_WIDE_ACCUM_MAX: return g_opt_wide_accum_max;
        case SIPP_OPT_BATCH_KPG_MAX: return g_opt_batch_kpg_max;
        case SIPP_OPT_FOLD_STRAUS: return g_opt_fold_straus;
        case SIPP_OPT_BATCH_STREAMS: return g_opt_batch_streams;
        case SIPP_OPT_BATCH_QLINES: return g_opt_batch_qlines;
        case SIPP_OPT_VALIDATE_POINTS: return g_opt_validate;
        case SIPP_OPT_PRODUCT_CHUNK_PAIRS: return g_opt_product_chunk;
        case SIPP_OPT_MATRIX_TAIL: return g_opt_matrix_n;
        case SIPP_OPT_MATRIX_FIRST: return g_opt_matrix_first;
        case SIPP_OPT_MATRIX_BLOCK_N: return g_opt_matrix_block_n;
        case SIPP_OPT_MATRIX_BLOCK_R: return g_opt_matrix_block_r;
        default: return -1;
    }
}

int sipp_get_stats(sipp_stats* out) {
    if (!out) return fail(SIPP_ERR_ARG, "null stats");
    if (g_device >= 0) collect_spans();
    *out = g_stats;
    return SIPP_OK;
}
int sipp_reset_stats(void) {
    if (g_device >= 0) collect_spans();
    memset(&g_stats, 0, sizeof g_stats);
    return SIPP_OK;
}

// ------------------------------------------------------------------------------------------------ contexts
// `defer`: the on-curve / subgroup check (1.35 ms of pure latency at any size: one 63-bit scalar multiplication per thread) runs on
// the side stream next to the prover's first kernels instead of in front of them; the whole-protocol entry points collect its
// verdict with ctx_finish_validation before they return anything, and the first in-place fold waits for it.
static int ctx_create_from_device_ex(const void* dA, const void* dB, size_t n, sipp_ctx** out, bool defer) {
    int rc = ensure_init();
    if (rc) return rc;
    if (!dA || !dB || !out || n == 0) return fail(SIPP_ERR_ARG, "sipp_ctx_create: null pointer or n == 0");
    rc = scratch_reserve(1);
    if (rc) return rc;
    sipp_ctx* c;
    rc = ctx_alloc(n, &c);
    if (rc) return rc;
    launch_decode((const uint32_t*)dA, c->dA, n * 2, g_stream, true);
    launch_codec_decode((const uint32_t*)dB, c->dB, n * 4, g_scr.flag, g_stream);
    g_stats.launches++;
    cudaError_t e = cudaSuccess;
    if (g_opt_validate) {
        // what G1Affine::new / G2Affine::new assert in the reference: on the curve, in the prime-order subgroup (the folds use
        // the endomorphisms, which are [lambda] / [6x^2] only there)
        if (defer) {
            if (!g_fold_stream) e = cudaStreamCreateWithFlags(&g_fold_stream, cudaStreamNonBlocking);
            if (e == cudaSuccess) e = order_after(g_fold_stream, g_stream);
            if (e == cudaSuccess) e = cudaMemsetAsync(g_scr.vflag, 0, sizeof(int), g_fold_stream);
            if (e == cudaSuccess) {
                Span sp(3, g_fold_stream);
                launch_validate_points(c->dA, c->dB, n, g_scr.vflag, g_fold_stream);
            }
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->validated, cudaEventDisableTiming);
            if (e == cudaSuccess) e = cudaEventRecord(c->validated, g_fold_stream);
            c->pending_validation = e == cudaSuccess;
        } else {
            Span sp(3, g_stream);
            launch_validate_points(c->dA, c->dB, n, g_scr.flag, g_stream);
        }
        g_stats.launches++;
    }
    int flag = 0;
    if (e == cudaSuccess) e = cudaMemcpyAsync(&flag, g_scr.flag, sizeof(int), cudaMemcpyDeviceToHost, g_stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(g_stream);
    if (e != cudaSuccess) { sipp_ctx_destroy(c); return cuda_fail(e, "decode"); }
    if (flag) {
        sipp_ctx_destroy(c);
        return fail(SIPP_ERR_ENCODING, (flag & 1) ? "input coordinate >= p" : (flag & 2) ? "input point is not on the curve"
                                                                                         : "input G2 point is not in the prime-order subgroup");
    }
    *out = c;
    return SIPP_OK;
}
int sipp_ctx_create_from_device(const void* dA, const void* dB, size_t n, sipp_ctx** out) { return ctx_create_from_device_ex(dA, dB, n, out, false); }

// the verdict of a deferred validation (SIPP_OK when there was none)
static int ctx_finish_validation(sipp_ctx* c) {
    if (!c || !c->pending_validation) return SIPP_OK;
    c->pending_validation = false;
    int flag = 0;
    cudaError_t e = cudaEventSynchronize(c->validated);
    if (e == cudaSuccess) e = cudaMemcpy(&flag, g_scr.vflag, sizeof(int), cudaMemcpyDeviceToHost);
    cudaEventDestroy(c->validated);
    c->validated = nullptr;
    if (e != cudaSuccess) return cuda_fail(e, "point validation");
    if (flag) return fail(SIPP_ERR_ENCODING, (flag & 2) ? "input point is not on the curve" : "input G2 point is not in the prime-order subgroup");
    return SIPP_OK;
}

static int ctx_create_ex(const uint8_t* A, const uint8_t* B, size_t n, sipp_ctx** out, bool defer);
static int ctx_create_ex(const uint8_t* A, const uint8_t* B, size_t n, sipp_ctx** out, bool defer) {
    int rc = ensure_init();
    if (rc) return rc;
    if (!A || !B || !out || n == 0) return fail(SIPP_ERR_ARG, "sipp_ctx_create: null pointer or n == 0");
    uint8_t *tA = nullptr, *tB = nullptr;
    CK(pool_alloc((void**)&tA, n * 64));
    cudaError_t e = pool_alloc((void**)&tB, n * 128);
    if (e != cudaSuccess) { pool_free(tA); return cuda_fail(e, "cudaMalloc"); }
    e = cudaMemcpyAsync(tA, A, n * 64, cudaMemcpyHostToDevice, g_stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(tB, B, n * 128, cudaMemcpyHostToDevice, g_stream);
    if (e != cudaSuccess) { pool_free(tA); pool_free(tB); return cuda_fail(e, "H2D"); }
    rc = ctx_create_from_device_ex(tA, tB, n, out, defer);  // synchronises the stream: the staging blocks are idle on return
    pool_free(tA);
    pool_free(tB);
    return rc;
}

int sipp_ctx_create(const uint8_t* A, const uint8_t* B, size_t n, sipp_ctx** out) { return ctx_create_ex(A, B, n, out, false); }

int sipp_ctx_destroy(sipp_ctx* c) {
    if (!c) return SIPP_OK;
    if (c->pending_validation) {  // the side stream still reads the points
        cudaEventSynchronize(c->validated);
        cudaEventDestroy(c->validated);
        c->pending_validation = false;
    }
    // every entry point that enqueues work on a context synchronises before returning results, and a block handed
    // out again is only touched by later work on the same stream, so recycling without a device sync is safe
    pool_free(c->dA);
    pool_free(c->dB);
    delete c;
    g_live_ctx--;
    return SIPP_OK;
}

size_t sipp_ctx_len(const sipp_ctx* c) { return c ? c->n : 0; }

int sipp_ctx_set_stages(sipp_ctx* c, int on) {
    if (!c) return fail(SIPP_ERR_ARG, "null ctx");
    if (c->mt.n) return fail(SIPP_ERR_ARG, "a pairing-matrix stage is in progress");
    c->stages = on != 0;
    return SIPP_OK;
}

int sipp_ctx_inner_product(sipp_ctx* c, uint8_t out[384]) {
    if (!c || !out) return fail(SIPP_ERR_ARG, "null argument");
    if (c->stages && !c->mt.n) {
        if (const size_t nr0 = mat_stage_first(c->n)) {  // Z and the first rounds from ONE matrix over the inputs
            int rc = mat_build(c, c->mt, nr0);
            return rc ? rc : mat_diag_product(c->mt, out);
        }
    }
    return ctx_products(c, 0, out, nullptr);
}

int sipp_ctx_cross_products(sipp_ctx* c, uint8_t zl[384], uint8_t zr[384]) {
    if (!c || !zl || !zr) return fail(SIPP_ERR_ARG, "null argument");
    if (c->stages) {
        if (c->n < 2) return fail(SIPP_ERR_ARG, "cross products need n >= 2");
        if (!c->mt.n) {
            const size_t nr = mat_stage(c->n);  // a pairing-matrix stage starts here?
            if (nr) {
                int rc = mat_build(c, c->mt, nr);
                if (rc) return rc;
            }
        }
        if (c->mt.n) return mat_products(c->mt, zl, zr);
    }
    return ctx_products(c, 1, zl, zr);
}

int sipp_ctx_fold(sipp_ctx* c, const uint8_t x[32], const uint8_t x_inv[32]) {
    if (!c || !x || !x_inv) return fail(SIPP_ERR_ARG, "null argument");
    if (int rc = check_fold_scalars(x, x_inv)) return rc;  // before any stage dispatch or device work: a refusal changes nothing
    if (c->n < 2) return fail(SIPP_ERR_ARG, "fold needs n >= 2");
    if (c->pending_validation) CK(cudaStreamWaitEvent(g_stream, c->validated, 0));  // the deferred check reads the points folded here
    if (c->mt.n) return mat_fold(c, c->mt, x, x_inv);  // :60-74 on the matrix of the stage in progress
    size_t h = c->n / 2;
    FoldPlan plan;
    if (fold_plan_build(x, x_inv, &plan)) return fail(SIPP_ERR_ENCODING, "fold scalar out of range (must be < r)");
    {
        Span sp(2, g_stream);
        // new_A = a1 + a2.mul(x)  prover_native.rs:60-64;  new_B = b1 + b2.mul(inv_x)  :65-69
        int e;
        if (g_opt_fold_straus && h >= 16384) {
            // a launch that fills the GPU: one thread per element, doublings shared by the components (k_fold_straus reads the plan
            // from device memory: the batched prover has one per instance)
            if (!g_fold_plan_dev) CK(cudaMalloc(&g_fold_plan_dev, sizeof(FoldPlan)));
            FoldPlan* d_plan = g_fold_plan_dev;
            CK(cudaMemcpyAsync(d_plan, &plan, sizeof plan, cudaMemcpyHostToDevice, g_stream));  // pageable source: staged before the call returns
            e = launch_fold_straus(c->dA, c->dB, h, c->n, 1, d_plan, g_stream);
        } else {
            e = h <= (size_t)g_opt_wide_fold_max ? launch_fold_wide(c->dA, c->dB, h, plan, g_stream) : launch_fold(c->dA, c->dB, h, plan, g_stream);
        }
        if (e) return cuda_fail((cudaError_t)e, "k_fold");
    }
    g_stats.launches += 1;
    g_stats.fold_points += h;
    c->n = h;                                                                       // n = n / 2   :74
    return SIPP_OK;
}

int sipp_ctx_read(sipp_ctx* c, uint8_t* A_out, uint8_t* B_out) {
    if (!c) return fail(SIPP_ERR_ARG, "null ctx");
    if (c->stale) return fail(SIPP_ERR_ARG, "the points of this context were not folded during its pairing-matrix tail (sipp_ctx_set_stages)");
    if (c->mt.n && c->mt.fold_points) CK(order_after(g_stream, g_fold_stream));  // look-ahead stage: the folds run on the side stream
    size_t n = c->n;
    uint32_t* tmp;
    CK(pool_alloc((void**)&tmp, n * 32 * sizeof(uint32_t)));
    cudaError_t e = cudaSuccess;
    if (A_out) {
        launch_codec_encode(c->dA, tmp, n * 2, g_stream);
        g_stats.launches++;
        e = cudaMemcpyAsync(A_out, tmp, n * 64, cudaMemcpyDeviceToHost, g_stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(g_stream);
    }
    if (B_out && e == cudaSuccess) {
        launch_codec_encode(c->dB, tmp, n * 4, g_stream);
        g_stats.launches++;
        e = cudaMemcpyAsync(B_out, tmp, n * 128, cudaMemcpyDeviceToHost, g_stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(g_stream);
    }
    pool_free(tmp);
    if (e != cudaSuccess) return cuda_fail(e, "sipp_ctx_read");
    return SIPP_OK;
}

// ------------------------------------------------------------------------------------------------ multi-GPU pieces
int sipp_ctx_partial_products(sipp_ctx* c, int which, void* d_out, void* stream) {
    if (!c || !d_out) return fail(SIPP_ERR_ARG, "null argument");
    // NULL is the legacy default stream (what torch.cuda.current_stream().cuda_stream is unless the caller switched
    // streams) -- NOT the library stream: g_stream is non-blocking and does not synchronise with it implicitly.
    cudaStream_t s = stream ? (cudaStream_t)stream : cudaStreamLegacy;
    // the caller's stream (e.g. torch's current stream, which NCCL orders against) must see the folds issued on the
    // library stream, and later library work must see these launches
    if (s != g_stream) CK(order_after(s, g_stream));
    size_t blocks;
    int nprod;
    int rc = ctx_products_to_device(c, which, &blocks, &nprod, s);
    if (rc) return rc;
    rc = launch_reduce(g_scr.partials, (int)blocks, nprod, (uint32_t*)d_out, false, s);
    if (rc) return rc;
    if (s != g_stream) CK(order_after(g_stream, s));
    return SIPP_OK;
}

int sipp_combine_partials(const void* d_partials, int count, int nprod, uint8_t* out, void* stream) {
    int rc = ensure_init();
    if (rc) return rc;
    if (!d_partials || !out || count < 1 || nprod < 1 || nprod > 2) return fail(SIPP_ERR_ARG, "bad argument");
    rc = scratch_reserve(1);
    if (rc) return rc;
    cudaStream_t s = stream ? (cudaStream_t)stream : cudaStreamLegacy;  // NULL = legacy default stream (see above)
    if (s != g_stream) CK(order_after(s, g_stream));
    rc = launch_reduce((const uint32_t*)d_partials, count, nprod, g_scr.out, true, s);
    if (rc) return rc;
    CK(cudaMemcpyAsync(g_scr.h_out, g_scr.out, (size_t)nprod * 384, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    memcpy(out, g_scr.h_out, (size_t)nprod * 384);
    return SIPP_OK;
}

// ------------------------------------------------------------------------------------------------ stand-alone
int sipp_inner_product(const uint8_t* A, const uint8_t* B, size_t n, uint8_t out[384]) {
    if (!out) return fail(SIPP_ERR_ARG, "null argument");
    if (n == 0) {  // fold(Fq12::one(), ...) over an empty iterator
        memset(out, 0, 384);
        out[0] = 1;
        return ensure_init();
    }
    sipp_ctx* c;
    int rc = sipp_ctx_create(A, B, n, &c);
    if (rc) return rc;
    rc = sipp_ctx_inner_product(c, out);
    sipp_ctx_destroy(c);
    return rc;
}

int sipp_pairing(const uint8_t a[64], const uint8_t b[128], uint8_t out[384]) { return sipp_inner_product(a, b, 1, out); }

int sipp_gt_fold(const uint8_t zl[384], const uint8_t z[384], const uint8_t zr[384], const uint8_t x[32], const uint8_t x_inv[32],
                 uint8_t out[384]) {
    if (!zl || !z || !zr || !x || !x_inv || !out) return fail(SIPP_ERR_ARG, "null argument");
    int rc = check_fold_scalars(x, x_inv);  // raw 256-bit exponents: x and x + r differ on an Fq12 outside GT
    if (rc) return rc;
    rc = ensure_init();
    if (rc) return rc;
    rc = scratch_reserve(1);
    if (rc) return rc;
    uint32_t* d_in;
    CK(cudaMalloc(&d_in, 3 * 384));
    cudaMemcpyAsync(d_in, zl, 384, cudaMemcpyHostToDevice, g_stream);
    cudaMemcpyAsync(d_in + 96, z, 384, cudaMemcpyHostToDevice, g_stream);
    cudaMemcpyAsync(d_in + 192, zr, 384, cudaMemcpyHostToDevice, g_stream);
    {
        Span sp(3, g_stream);
        // two 32-lane Fq12 machines, one power each (k_gt_fold_eng); the one-thread-per-power kernel stays as the engines-off arm
        if (g_opt_fe_engine) launch_gt_fold_eng(d_in, scalar_from_bytes(x), scalar_from_bytes(x_inv), g_scr.out, g_stream);
        else launch_gt_fold(d_in, scalar_from_bytes(x), scalar_from_bytes(x_inv), g_scr.out, g_stream);
    }
    g_stats.launches++;
    cudaError_t e = cudaMemcpyAsync(g_scr.h_out, g_scr.out, 384, cudaMemcpyDeviceToHost, g_stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(g_stream);
    cudaFree(d_in);
    if (e != cudaSuccess) return cuda_fail(e, "sipp_gt_fold");
    memcpy(out, g_scr.h_out, 384);
    return SIPP_OK;
}

// Fr inverse on the host (one per round; prover_native.rs:58): the binary extended Euclid of glv_core.h, the same code the
// device transcript runs per instance (a few microseconds; x^(r-2) took 15)
int sipp_fr_inverse(const uint8_t x[32], uint8_t out[32]) {
    if (!x || !out) return fail(SIPP_ERR_ARG, "null argument");
    uint64_t v[4], r[4] = {0, 0, 0, 0};
    memcpy(v, x, 32);
    const int rc = sipp::glv::fr_inverse_binary(v, r);
    if (rc == -1) return fail(SIPP_ERR_ENCODING, "scalar >= r");
    if (rc == -2) return fail(SIPP_ERR_ZERO_CHALLENGE, "challenge is zero: x.inverse().unwrap() panics in the reference");
    memcpy(out, r, 32);
    return SIPP_OK;
}

// ------------------------------------------------------------------------------------------------ protocol
size_t sipp_proof_len(size_t n) { return is_pow2(n) ? 2 * log2_exact(n) + 1 : 0; }

// the protocol loop on a context whose A, B are being absorbed by `job` (started by the caller as early as possible)
}  // extern "C"
namespace sipp_host {
int prove_core(sipp_ctx* c, AbsorbJob& job, uint8_t* proof) {
    size_t n = c->n;
    size_t np = sipp_proof_len(n);
    std::vector<uint8_t> fwd(np * 384);  // proof in push order; reversed at the end (prover_native.rs:78)
    size_t k = 0;
    sipp_transcript& tr = job.tr;
    c->stages = true;  // Z_L, Z_R and the folds may come from pairing-matrix stages (same values; k_mat.cu)
    int rc = sipp_ctx_inner_product(c, &fwd[384 * k]);                       // let Z = inner_product(A, B);   :29
    k++;
    bool first = true;
    while (rc == SIPP_OK && n > 1) {                                          // :45
        uint8_t* zl = &fwd[384 * k];
        uint8_t* zr = &fwd[384 * (k + 1)];
        rc = sipp_ctx_cross_products(c, zl, zr);                              // :46-49
        if (rc) break;
        if (first) {
            g_stats.transcript_ms += job.join();                              // :36-39 finished? (exposed wait only)
            sipp_transcript_append_fq12(&tr, &fwd[0]);                        // proof.push(Z); transcript.append_fq12(Z)  :42-43
            first = false;
        }
        auto h0 = std::chrono::steady_clock::now();
        sipp_transcript_append_fq12(&tr, zl);                                 // :52-53
        sipp_transcript_append_fq12(&tr, zr);                                 // :54-55
        k += 2;
        uint8_t x[32], xinv[32];
        sipp_transcript_get_challenge(&tr, x);                                // :57
        rc = sipp_fr_inverse(x, xinv);                                        // :58
        g_stats.transcript_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - h0).count();
        if (rc) break;
        rc = sipp_ctx_fold(c, x, xinv);                                       // :60-74
        n = c->n;
    }
    if (rc) return rc;
    for (size_t i = 0; i < np; i++) memcpy(proof + 384 * i, &fwd[384 * (np - 1 - i)], 384);  // proof.reverse()  :78
    return SIPP_OK;
}
}  // namespace sipp_host
extern "C" {

int sipp_ctx_prove(sipp_ctx* c, const uint8_t* A, const uint8_t* B, uint8_t* proof) {
    if (!c || !A || !B || !proof) return fail(SIPP_ERR_ARG, "null argument");
    if (!is_pow2(c->n)) return fail(SIPP_ERR_ARG, "n must be a power of two (the reference halves n every round)");
    // register A and B (prover_native.rs:36-39): a strictly serial 8n-permutation hash chain.  It does not depend on
    // anything the GPU computes, so it runs on a host thread while the GPU computes Z and the first Z_L, Z_R.
    AbsorbJob job;
    job.start(A, B, c->n);
    return prove_core(c, job, proof);
}

int sipp_prove_native(const uint8_t* A, size_t a_len, const uint8_t* B, size_t b_len, uint8_t* proof) {
    if (a_len != b_len) return fail(SIPP_ERR_LENGTH, "assert_eq!(A.len(), B.len()) failed");  // prover_native.rs:27
    if (!is_pow2(a_len)) return fail(SIPP_ERR_ARG, "n must be a non-zero power of two");
    if (!A || !B || !proof) return fail(SIPP_ERR_ARG, "null argument");
    int rc = ensure_init();
    if (rc) return rc;
    // the hash chain starts before the upload: the H2D copies, the decode and the point validation run in its shadow
    AbsorbJob job;
    job.start(A, B, a_len);
    sipp_ctx* c;
    rc = ctx_create_ex(A, B, a_len, &c, true);  // the point validation runs beside the first kernels; its verdict is collected below
    if (rc) return rc;
    rc = prove_core(c, job, proof);
    const int vrc = ctx_finish_validation(c);
    sipp_ctx_destroy(c);
    return vrc ? vrc : rc;
}

int sipp_verify_native(const uint8_t* A, size_t a_len, const uint8_t* B, size_t b_len, const uint8_t* proof, size_t proof_len, uint8_t* final_A,
                       uint8_t* final_B, uint8_t* final_Z) {
    if (!A || !B || !proof) return fail(SIPP_ERR_ARG, "null argument");
    if (a_len != b_len) return fail(SIPP_ERR_LENGTH, "A.len() != B.len()");
    size_t n = a_len;
    if (!is_pow2(n)) return fail(SIPP_ERR_ARG, "n must be a non-zero power of two");
    if (proof_len < sipp_proof_len(n)) return fail(SIPP_ERR_SHORT_PROOF, "proof.pop().unwrap() on an empty proof");  // verifier_native.rs:31,40,42
    // an Fq12 the reference could not have deserialised (a coordinate >= p) is refused, as for A and B
    if (!fq_bytes_canonical(proof + 384 * (proof_len - sipp_proof_len(n)), 12 * sipp_proof_len(n))) return fail(SIPP_ERR_ENCODING, "proof coordinate >= p");
    int rc = ensure_init();
    if (rc) return rc;
    // :25-28 on a host thread while the GPU receives, decodes and validates A, B (nothing else can overlap: the first fold needs
    // the first challenge, which needs the whole chain)
    AbsorbJob job;
    job.start(A, B, n);
    sipp_ctx* c;
    rc = ctx_create_ex(A, B, n, &c, true);  // point validation beside the transcript replay; verdict collected before the result
    if (rc) return rc;
    g_stats.transcript_ms += job.join();
    sipp_transcript& tr = job.tr;
    size_t top = proof_len;
    uint8_t Z[384];
    memcpy(Z, proof + 384 * --top, 384);                                      // let original_Z = proof.pop().unwrap();  :31
    sipp_transcript_append_fq12(&tr, Z);                                      // :33
    // The challenges depend only on A, B and the proof (:33-45): replay the transcript first, then every fold is queued back to
    // back and every GT update Z_L^x, Z_R^(1/x) (:59-61) is an independent power -- all of them in ONE launch on the side stream.
    const size_t rounds = log2_exact(n);
    std::vector<uint8_t> xs(rounds * 64), elems((2 * rounds + 1) * 384);
    memcpy(elems.data(), Z, 384);
    for (size_t k = 0; k < rounds && !rc; k++) {                              // :35
        const uint8_t* zl = proof + 384 * --top;                              // :40
        sipp_transcript_append_fq12(&tr, zl);
        const uint8_t* zr = proof + 384 * --top;                              // :42
        sipp_transcript_append_fq12(&tr, zr);
        sipp_transcript_get_challenge(&tr, &xs[64 * k]);                      // :45
        rc = sipp_fr_inverse(&xs[64 * k], &xs[64 * k + 32]);                  // :46
        memcpy(&elems[384 * (1 + 2 * k)], zl, 384);
        memcpy(&elems[384 * (2 + 2 * k)], zr, 384);
    }
    uint32_t *d_elems = nullptr, *d_xs = nullptr, *d_parts = nullptr, *d_z = nullptr;
    const bool gt_batched = !rc && rounds > 0 && g_opt_fe_engine;
    if (gt_batched) {
        if (!g_fold_stream) CK(cudaStreamCreateWithFlags(&g_fold_stream, cudaStreamNonBlocking));
        cudaError_t e = pool_alloc((void**)&d_elems, elems.size());
        if (e == cudaSuccess) e = pool_alloc((void**)&d_xs, xs.size());
        if (e == cudaSuccess) e = pool_alloc((void**)&d_parts, (rounds + 1) * 384);
        if (e == cudaSuccess) e = pool_alloc((void**)&d_z, 384);
        if (e == cudaSuccess) e = order_after(g_fold_stream, g_stream);      // pool blocks: earlier users ran on the library stream
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_elems, elems.data(), elems.size(), cudaMemcpyHostToDevice, g_fold_stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_xs, xs.data(), xs.size(), cudaMemcpyHostToDevice, g_fold_stream);
        int le = 0;
        if (e == cudaSuccess) {
            Span sp(3, g_fold_stream);
            le = launch_gt_fold_rounds(d_elems, d_xs, (int)rounds, d_parts, g_fold_stream);
            if (!le) le = launch_reduce_fe_eng(d_parts, (int)rounds + 1, 1, d_z, 2, g_opt_fe_norm, g_fold_stream);
            g_stats.launches += 2;
        }
        if (e == cudaSuccess && !le) e = cudaMemcpyAsync(Z, d_z, 384, cudaMemcpyDeviceToHost, g_fold_stream);  // Z: pageable, synchronised below
        if (e != cudaSuccess || le) {
            cudaStreamSynchronize(g_fold_stream);
            pool_free(d_elems); pool_free(d_xs); pool_free(d_parts); pool_free(d_z);
            sipp_ctx_destroy(c);
            return e != cudaSuccess ? cuda_fail(e, "verifier GT updates") : cuda_fail((cudaError_t)le, "k_gt_fold_rounds");
        }
    }
    for (size_t k = 0; k < rounds && !rc; k++) {
        rc = sipp_ctx_fold(c, &xs[64 * k], &xs[64 * k + 32]);                 // :48-57
        if (!rc && !gt_batched) {
            uint8_t nz[384];
            rc = sipp_gt_fold(&elems[384 * (1 + 2 * k)], Z, &elems[384 * (2 + 2 * k)], &xs[64 * k], &xs[64 * k + 32], nz);  // :59-61
            if (!rc) memcpy(Z, nz, 384);
        }
    }
    n = c->n;
    if (gt_batched) {
        cudaError_t e = cudaStreamSynchronize(g_fold_stream);
        pool_free(d_elems); pool_free(d_xs); pool_free(d_parts); pool_free(d_z);
        if (e != cudaSuccess) { sipp_ctx_destroy(c); return cuda_fail(e, "verifier GT updates"); }
    }
    uint8_t fa[64], fb[128], e[384];
    if (!rc) rc = sipp_ctx_read(c, fa, fb);                                   // final_A: A[0], final_B: B[0]   :74-75
    if (!rc) rc = sipp_ctx_inner_product(c, e);                               // pairing(final_A, final_B)      :80
    const int vrc = ctx_finish_validation(c);                                 // G1Affine::new / G2Affine::new of the inputs
    sipp_ctx_destroy(c);
    if (vrc) return vrc;
    if (rc) return rc;
    if (final_A) memcpy(final_A, fa, 64);
    if (final_B) memcpy(final_B, fb, 128);
    if (final_Z) memcpy(final_Z, Z, 384);
    if (memcmp(e, Z, 384) != 0) return fail(SIPP_ERR_VERIFY, "Verification failed");  // :81-84
    return SIPP_OK;
}

// ------------------------------------------------------------------------------------------------ test hooks
int sipp_test_fq_op(int op, const uint8_t* a, const uint8_t* b, uint8_t* out, size_t count) {
    int rc = ensure_init();
    if (rc) return rc;
    if (!a || !out || count == 0) return fail(SIPP_ERR_ARG, "bad argument");
    uint32_t *da, *db = nullptr, *dout;
    CK(cudaMalloc(&da, count * 32));
    CK(cudaMalloc(&dout, count * 32));
    if (b) { CK(cudaMalloc(&db, count * 32)); CK(cudaMemcpyAsync(db, b, count * 32, cudaMemcpyHostToDevice, g_stream)); }
    CK(cudaMemcpyAsync(da, a, count * 32, cudaMemcpyHostToDevice, g_stream));
    launch_test_fq_op(op, da, db, dout, count, g_stream);
    g_stats.launches++;
    cudaError_t e = cudaStreamSynchronize(g_stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(out, dout, count * 32, cudaMemcpyDeviceToHost, g_stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(g_stream);
    cudaFree(da); cudaFree(dout); if (db) cudaFree(db);
    if (e != cudaSuccess) return cuda_fail(e, "sipp_test_fq_op");
    return SIPP_OK;
}

int sipp_test_fq12_op(int op, const uint8_t* a, const uint8_t* b, uint8_t* out, size_t count) {
    int rc = ensure_init();
    if (rc) return rc;
    if (!a || !out || count == 0) return fail(SIPP_ERR_ARG, "bad argument");
    uint32_t *da, *db = nullptr, *dout;
    CK(cudaMalloc(&da, count * 384));
    CK(cudaMalloc(&dout, count * 384));
    if (b) { CK(cudaMalloc(&db, count * 384)); CK(cudaMemcpyAsync(db, b, count * 384, cudaMemcpyHostToDevice, g_stream)); }
    CK(cudaMemcpyAsync(da, a, count * 384, cudaMemcpyHostToDevice, g_stream));
    if (op >= 20) launch_test_coop_op(op - 20, da, db, dout, count, g_stream);
    else launch_test_fq12_op(op, da, db, dout, count, g_stream);
    g_stats.launches++;
    cudaError_t e = cudaStreamSynchronize(g_stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(out, dout, count * 384, cudaMemcpyDeviceToHost, g_stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(g_stream);
    cudaFree(da); cudaFree(dout); if (db) cudaFree(db);
    if (e != cudaSuccess) return cuda_fail(e, "sipp_test_fq12_op");
    return SIPP_OK;
}

int sipp_test_fold_plan(const uint8_t x[32], const uint8_t x_inv[32], uint32_t* out_words, size_t out_cap) {
    if (!x || !x_inv || !out_words || out_cap < sizeof(FoldPlan) / 4) return fail(SIPP_ERR_ARG, "bad argument");
    FoldPlan plan;
    if (fold_plan_build(x, x_inv, &plan)) return fail(SIPP_ERR_ENCODING, "fold scalar out of range (must be < r)");
    memcpy(out_words, &plan, sizeof plan);
    return (int)(sizeof(FoldPlan) / 4);
}

int sipp_test_fold_plan_device(const uint8_t* x, const uint8_t* x_inv, size_t count, uint32_t* out_words) {
    if (!x || !x_inv || !out_words || count == 0) return fail(SIPP_ERR_ARG, "bad argument");
    int rc = ensure_init();
    if (rc) return rc;
    uint64_t *dx = nullptr, *dxi = nullptr;
    FoldPlan* dplans = nullptr;
    int* dfails = nullptr;
    int fails = 0;
    cudaError_t e = cudaMalloc(&dx, count * 32);
    if (e == cudaSuccess) e = cudaMalloc(&dxi, count * 32);
    if (e == cudaSuccess) e = cudaMalloc(&dplans, count * sizeof(FoldPlan));
    if (e == cudaSuccess) e = cudaMalloc(&dfails, sizeof(int));
    if (e == cudaSuccess) e = cudaMemcpyAsync(dx, x, count * 32, cudaMemcpyHostToDevice, g_stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(dxi, x_inv, count * 32, cudaMemcpyHostToDevice, g_stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(dfails, 0, sizeof(int), g_stream);
    if (e == cudaSuccess) e = (cudaError_t)launch_test_plan_build(dx, dxi, count, dplans, dfails, g_stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(out_words, dplans, count * sizeof(FoldPlan), cudaMemcpyDeviceToHost, g_stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(&fails, dfails, sizeof(int), cudaMemcpyDeviceToHost, g_stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(g_stream);
    g_stats.launches++;
    cudaFree(dx); cudaFree(dxi); cudaFree(dplans); cudaFree(dfails);
    if (e != cudaSuccess) return cuda_fail(e, "sipp_test_fold_plan_device");
    return fails;
}

int sipp_test_fold_batch(const uint8_t* A, const uint8_t* B, size_t n, size_t count, const uint8_t* xs, const uint8_t* x_invs, int kernel,
                         uint8_t* A_out, uint8_t* B_out) {
    if (!A || !B || !xs || !x_invs || !A_out || !B_out || count == 0 || n < 2 || n % 2 || kernel < 0 || kernel > 2)
        return fail(SIPP_ERR_ARG, "bad argument");
    std::vector<FoldPlan> plans(count);
    for (size_t j = 0; j < count; j++) {
        int rc = check_fold_scalars(xs + 32 * j, x_invs + 32 * j);
        if (rc) return rc;
        if (fold_plan_build(xs + 32 * j, x_invs + 32 * j, &plans[j])) return fail(SIPP_ERR_ENCODING, "fold scalar out of range (must be < r)");
    }
    sipp_ctx* c;
    int rc = ctx_create_ex(A, B, n * count, &c, false);  // decode + point checks as sipp_ctx_create
    if (rc) return rc;
    const size_t h = n / 2, total = n * count;
    FoldPlan* dplans = nullptr;
    cudaError_t e = pool_alloc((void**)&dplans, count * sizeof(FoldPlan));
    if (e == cudaSuccess) e = cudaMemcpyAsync(dplans, plans.data(), count * sizeof(FoldPlan), cudaMemcpyHostToDevice, g_stream);
    if (e == cudaSuccess) {
        Span sp(2, g_stream);
        e = (cudaError_t)(kernel == 0   ? launch_fold_batch(c->dA, c->dB, h, n, count, dplans, g_stream)
                          : kernel == 1 ? launch_fold_wide_batch(c->dA, c->dB, h, n, count, dplans, g_stream)
                                        : launch_fold_straus(c->dA, c->dB, h, n, count, dplans, g_stream));
        g_stats.launches++;
    }
    std::vector<uint8_t> a(total * 64), b(total * 128);
    if (e == cudaSuccess) e = cudaStreamSynchronize(g_stream);  // the plans were staged from pageable memory
    pool_free(dplans);
    if (e != cudaSuccess) { sipp_ctx_destroy(c); return cuda_fail(e, "sipp_test_fold_batch"); }
    rc = sipp_ctx_read(c, a.data(), b.data());
    sipp_ctx_destroy(c);
    if (rc) return rc;
    for (size_t j = 0; j < count; j++) {
        memcpy(A_out + 64 * h * j, &a[64 * n * j], 64 * h);
        memcpy(B_out + 128 * h * j, &b[128 * n * j], 128 * h);
    }
    return SIPP_OK;
}

int sipp_microbench(int which, int iters, double* ops_per_s, double* ms_out) {
    int rc = ensure_init();
    if (rc) return rc;
    if (!ops_per_s || iters < 1) return fail(SIPP_ERR_ARG, "bad argument");
    const int threads = 256;
    const int blocks = g_sm_count * 8;
    uint64_t* d_out;
    CK(cudaMalloc(&d_out, (size_t)blocks * threads * sizeof(uint64_t)));
    cudaEvent_t a, b;
    CK(cudaEventCreate(&a));
    CK(cudaEventCreate(&b));
    double per_thread_ops = 0;
    float best = 1e30f;
    for (int rep = 0; rep < 4; rep++) {  // first repetition is the warm-up
        CK(cudaEventRecord(a, g_stream));
        if (launch_microbench(which, blocks, threads, d_out, iters, 12345u + rep, &per_thread_ops, g_stream)) {
            cudaFree(d_out);
            return fail(SIPP_ERR_ARG, "unknown microbenchmark or launch failure");
        }
        g_stats.launches++;
        CK(cudaEventRecord(b, g_stream));
        CK(cudaEventSynchronize(b));
        float ms;
        CK(cudaEventElapsedTime(&ms, a, b));
        if (rep > 0 && ms < best) best = ms;
    }
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    cudaFree(d_out);
    *ops_per_s = per_thread_ops * threads * blocks / (best * 1e-3);
    if (ms_out) *ms_out = best;
    return SIPP_OK;
}

}  // extern "C"


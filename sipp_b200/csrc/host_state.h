// host_state.h -- process-wide host state of libsipp_b200 shared by its host translation units (sipp_b200.cu: the C ABI of the
// single proof; batch.cu: batched instances).  One host thread per process by contract, so none of this is locked.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include <atomic>
#include <thread>

#include "../../include/sipp_b200.h"
#include "launch.h"

namespace sipp_host {
void pool_free(void* p);
// A pairing-matrix stage of a single proof (k_mat.cu; SIPP_OPT_MATRIX_*): E[i][j] = <A_block_i, B_block_j> over the points of a
// context, then Z_L / Z_R as products of matrix entries and the fold as GT exponentiations of the matrix.
struct MatTail {
    uint32_t* E[2] = {nullptr, nullptr};
    int cur = 0;
    size_t n = 0;   // virtual points (blocks) the matrix stands for; 0 = no stage in progress
    size_t m = 1;   // points per block (1: the tail of the proof)
    bool fold_points = false;  // the points are still folded with every challenge (side stream): a later stage is built from them
    int folds = 0;  // point folds issued on the side stream in this stage
    void reset() {
        pool_free(E[0]);
        pool_free(E[1]);
        E[0] = E[1] = nullptr;
        n = 0;
        m = 1;
        fold_points = false;
    }
    ~MatTail() { reset(); }
};
}  // namespace sipp_host

// device-resident A, B of the current round of one prover (or one rank's strided shard of it)
struct sipp_ctx {
    uint32_t* dA = nullptr;  // n x 16 words, Montgomery
    uint32_t* dB = nullptr;  // n x 32 words
    size_t n = 0, cap = 0;
    bool stages = false;     // sipp_ctx_set_stages: products / folds may run on pairing-matrix stages
    bool stale = false;      // a tail stage ran: the points were not folded any more (sipp_ctx_read refuses)
    bool pending_validation = false;  // the on-curve / subgroup check of these points is still running on the side stream
    cudaEvent_t validated = nullptr;
    sipp_host::MatTail mt;
};

namespace sipp_host {

extern int g_device;             // CUDA device of this process, -1 before sipp_init
extern int g_sm_count;
extern cudaStream_t g_stream;    // the library's non-blocking stream
extern cudaStream_t g_fold_stream;  // its side stream (created on first use, sipp_b200.cu)
#define SIPP_FIRST_STAGE_LOG2_LOOPS 18
size_t mat_first_budget(size_t n);
extern int g_opt_pipeline, g_opt_fe_norm, g_opt_fq12_order, g_opt_profile, g_opt_fold_straus, g_opt_batch_kpg_max, g_opt_batch_streams, g_opt_batch_qlines, g_opt_wide_max, g_opt_wide_fold_max, g_opt_fe_engine, g_opt_validate, g_opt_matrix_n, g_opt_matrix_first, g_opt_matrix_block_n, g_opt_matrix_block_r, g_opt_product_chunk;
extern sipp_stats g_stats;

int fail(int code, const char* what);             // records the message for sipp_last_error, returns `code`
int cuda_fail(cudaError_t e, const char* what);   // same for a CUDA error, returns SIPP_ERR_CUDA
int ensure_init();
bool is_pow2(size_t n);

void batch_release_streams();   // batch.cu
// context with uninitialised device arrays for n points (pool blocks)
int ctx_alloc(size_t n, sipp_ctx** out);
// true when all `n_fq` little-endian 32-byte integers are < p (the canonical encoding ark-serialize requires: a proof element with a
// coordinate c + p would hash differently in the transcript while reducing to the same field element)
inline bool fq_bytes_canonical(const uint8_t* b, size_t n_fq) {
    static const uint64_t PM[4] = {0x3c208c16d87cfd47ull, 0x97816a916871ca8dull, 0xb85045b68181585dull, 0x30644e72e131a029ull};
    for (size_t i = 0; i < n_fq; i++) {
        uint64_t w[4];
        __builtin_memcpy(w, b + 32 * i, 32);
        bool less = false;
        for (int k = 3; k >= 0; k--) {
            if (w[k] != PM[k]) { less = w[k] < PM[k]; break; }
        }
        if (!less) return false;
    }
    return true;
}
// grow-only device memory pool (cudaFree synchronises the device; blocks are recycled, released in sipp_shutdown)
cudaError_t pool_alloc(void** out, size_t bytes);
// the line table shared by every Miller launch of the process (grow-only)
int lines_reserve(size_t bytes);
uint32_t* lines_buffer();
// make `later` wait for everything already enqueued on `earlier`
cudaError_t order_after(cudaStream_t later, cudaStream_t earlier);

// The registration of A and B in the transcript (prover_native.rs:36-39, verifier_native.rs:25-28): 8n strictly serial Poseidon
// permutations that depend on nothing the GPU computes, so they run on a host thread from the moment the inputs are known --
// under the upload, the decode + validation kernels, Z and the first Z_L / Z_R.  join() returns the milliseconds the caller
// had to wait (the exposed part of the chain).
struct AbsorbJob {
    sipp_transcript tr;
    std::thread th;
    std::atomic<bool> cancel{false};
    void start(const uint8_t* A, const uint8_t* B, size_t n) {
        sipp_transcript_new(&tr);
        th = std::thread([this, A, B, n]() {
            const size_t chunk = 512;
            for (size_t i = 0; i < n && !cancel.load(std::memory_order_relaxed); i += chunk)
                sipp_transcript_append_pairs(&tr, A + 64 * i, B + 128 * i, n - i < chunk ? n - i : chunk);
        });
    }
    double join();
    ~AbsorbJob() {
        cancel.store(true);
        if (th.joinable()) th.join();
    }
};

// pairing-matrix stages (sipp_b200.cu): used by the single-GPU prover and by rank 0's tail of the sharded one
size_t mat_stage_first(size_t n);  // blocks of the stage built from the inputs themselves (0: none)
int mat_diag_product(MatTail& mt, uint8_t* z);
size_t mat_stage(size_t n);  // number of blocks of the stage that starts with n points left (0: a plain round)
int mat_build(sipp_ctx* c, MatTail& mt, size_t nr);
int mat_build_ex(sipp_ctx* c, MatTail& mt, size_t nr, uint32_t* raw_out);
int mat_adopt(MatTail& mt, const uint32_t* gathered, int ranks, size_t nr);
int mat_products(MatTail& mt, uint8_t* zl, uint8_t* zr);
int mat_fold(sipp_ctx* c, MatTail& mt, const uint8_t x[32], const uint8_t xinv[32]);

// the protocol loop of a single GPU on a context whose A, B are being absorbed by `job` (sipp_b200.cu)
int prove_core(sipp_ctx* c, AbsorbJob& job, uint8_t* proof);

// CUDA-event span around a kernel class (SIPP_OPT_PROFILE): kind 0 miller, 1 reduce / final exponentiation, 2 fold, 3 other
int span_begin(int kind, cudaStream_t s);
void span_end(int idx, cudaStream_t s);
struct Span {
    int idx;
    cudaStream_t stream;
    Span(int kind, cudaStream_t s) : idx(span_begin(kind, s)), stream(s) {}
    ~Span() { span_end(idx, stream); }
};

}  // namespace sipp_host

#define CK(call)                                                    \
    do {                                                            \
        cudaError_t e_ = (call);                                    \
        if (e_ != cudaSuccess) return sipp_host::cuda_fail(e_, #call); \
    } while (0)

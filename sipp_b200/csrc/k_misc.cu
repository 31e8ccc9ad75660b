// k_misc.cu -- see kernels overview in device_common.cuh
#include "device_common.cuh"
#include "../../include/sipp_b200.h"

namespace sipp {

// ------------------------------------------------------------------------------------------------ codecs
// one thread per Fq element; `flags` (optional) receives 1 if any element was >= p
__global__ void k_codec_decode(const uint32_t* __restrict__ in, uint32_t* __restrict__ out, size_t n_fq, int* __restrict__ flags) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_fq) return;
    Fq c;
#pragma unroll
    for (int k = 0; k < 8; k++) c.l[k] = in[8 * i + k];
    const uint32_t P[8] = {SIPP_P0, SIPP_P1, SIPP_P2, SIPP_P3, SIPP_P4, SIPP_P5, SIPP_P6, SIPP_P7};
    uint32_t t[8];
    if (sub8(t, c.l, P) == 0 && flags) atomicOr(flags, 1);  // no borrow: value >= p
    Fq m = fq_to_mont(c);
#pragma unroll
    for (int k = 0; k < 8; k++) out[8 * i + k] = m.l[k];
}
__global__ void k_codec_encode(const uint32_t* __restrict__ in, uint32_t* __restrict__ out, size_t n_fq) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_fq) return;
    Fq m;
#pragma unroll
    for (int k = 0; k < 8; k++) m.l[k] = in[8 * i + k];
    Fq c = fq_from_mont(m);
#pragma unroll
    for (int k = 0; k < 8; k++) out[8 * i + k] = c.l[k];
}

// ------------------------------------------------------------------------------------------------ batched verifier outcome
// The per-instance outcome of the _device batched verifiers (batch.cu, ragged.cu), launched once the flags of the call were found
// clean.  One warp per instance j: the 12 np coordinates of its proof elements read, Fq12 [pt[j].first, pt[j].first + pt[j].np) of
// `proofs`, must all be < p (the host forms' fq_bytes_canonical) -- the lanes stride over the coordinates, one 32-byte little-endian
// integer each, and vote.  results[j] = SIPP_ERR_ENCODING when one is not, else SIPP_OK when z[j] == pair[j] (verifier_native.rs:81-84),
// else SIPP_ERR_VERIFY.  Then the finals that are non-NULL, unless the proof was not canonical and !enc_finals: final_Z[j] <- z[j],
// final_A[j] <- fin + 16 j, final_B[j] <- fin + 16 count + 32 j (words).
__global__ void __launch_bounds__(128) k_verify_outcome(const uint32_t* __restrict__ proofs, const RaggedProof* __restrict__ pt, size_t count,
                                                        const uint32_t* __restrict__ z, const uint32_t* __restrict__ pair,
                                                        const uint32_t* __restrict__ fin, int enc_finals, int* __restrict__ results,
                                                        uint32_t* __restrict__ final_A, uint32_t* __restrict__ final_B, uint32_t* __restrict__ final_Z) {
    const size_t j = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) / 32;
    const int lane = threadIdx.x & 31;
    if (j >= count) return;  // whole warps
    const RaggedProof t = pt[j];
    const uint32_t* e = proofs + 96 * t.first;
    const uint32_t P[8] = {SIPP_P0, SIPP_P1, SIPP_P2, SIPP_P3, SIPP_P4, SIPP_P5, SIPP_P6, SIPP_P7};
    bool ok = true;
    for (size_t c = lane; c < 12 * (size_t)t.np; c += 32) {
        uint32_t w[8], d[8];
#pragma unroll
        for (int k = 0; k < 8; k++) w[k] = e[8 * c + k];
        ok &= sub8(d, w, P) != 0;  // a borrow: w < p
    }
    const bool canonical = __all_sync(0xffffffffu, ok);
    bool same = true;
    for (int k = lane; k < 96; k += 32) same &= z[96 * j + k] == pair[96 * j + k];
    same = __all_sync(0xffffffffu, same);
    if (lane == 0) results[j] = !canonical ? SIPP_ERR_ENCODING : same ? SIPP_OK : SIPP_ERR_VERIFY;
    if (!canonical && !enc_finals) return;
    if (final_Z)
        for (int k = lane; k < 96; k += 32) final_Z[96 * j + k] = z[96 * j + k];
    if (final_A && lane < 16) final_A[16 * j + lane] = fin[16 * j + lane];
    if (final_B) final_B[32 * j + lane] = fin[16 * count + 32 * j + lane];
}

// ------------------------------------------------------------------------------------------------ test hooks
__global__ void k_test_fq_op(int op, const uint32_t* __restrict__ a, const uint32_t* __restrict__ b, uint32_t* __restrict__ out, size_t count) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    Fq x = fq_decode(a + 8 * i), y = b ? fq_decode(b + 8 * i) : fq_zero(), r;
    switch (op) {
        case 0: r = fq_mul(x, y); break;
        case 1: r = fq_mul_portable(x, y); break;
        case 2: r = fq_add(x, y); break;
        case 3: r = fq_sub(x, y); break;
        case 4: r = fq_inv(x); break;
        default: r = fq_neg(x); break;
    }
    fq_encode(out + 8 * i, r);
}
__global__ void __launch_bounds__(32) k_test_fq12_op(int op, const uint32_t* __restrict__ a, const uint32_t* __restrict__ b, uint32_t* __restrict__ out,
                                                     size_t count) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    Fq12 x = fq12_decode(a + 96 * i), r;
    Fq12 y = b ? fq12_decode(b + 96 * i) : fq12_one();
    switch (op) {
        case 0: r = fq12_mul(x, y); break;
        case 1: r = fq12_sqr(x); break;
        case 2: r = fq12_inv(x); break;
        case 3: r = fq12_frob(x, 1); break;
        case 4: r = fq12_frob(x, 2); break;
        case 5: r = fq12_frob(x, 3); break;
        case 6: r = fq12_conj(x); break;
        case 7: r = fq12_cyc_sqr(x); break;
        default: r = fq12_cyc_exp_x(x); break;
    }
    fq12_encode(out + 96 * i, r);
}

// ------------------------------------------------------------------------------------------------ microbenchmarks
// Each thread runs `iters` rounds of 8 independent dependent-chains; the result is stored so nothing is elided.
__global__ void __launch_bounds__(256) k_bench_mad_lo(uint32_t* out, int iters, uint32_t seed) {
    uint32_t a = seed + threadIdx.x, b = seed * 3 + blockIdx.x;
    uint32_t r0 = a, r1 = a + 1, r2 = a + 2, r3 = a + 3, r4 = a + 4, r5 = a + 5, r6 = a + 6, r7 = a + 7;
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int u = 0; u < 8; u++) {
            asm volatile("mad.lo.u32 %0, %0, %8, %9;\n\tmad.lo.u32 %1, %1, %8, %9;\n\tmad.lo.u32 %2, %2, %8, %9;\n\tmad.lo.u32 %3, %3, %8, %9;\n\t"
                         "mad.lo.u32 %4, %4, %8, %9;\n\tmad.lo.u32 %5, %5, %8, %9;\n\tmad.lo.u32 %6, %6, %8, %9;\n\tmad.lo.u32 %7, %7, %8, %9;"
                         : "+r"(r0), "+r"(r1), "+r"(r2), "+r"(r3), "+r"(r4), "+r"(r5), "+r"(r6), "+r"(r7)
                         : "r"(b), "r"(a));
        }
    }
    out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = r0 ^ r1 ^ r2 ^ r3 ^ r4 ^ r5 ^ r6 ^ r7;
}
// 8 x 8 schoolbook column accumulation with plain (carry-less) 32x32->64 multiply-adds whose operands change every
// round -- ptxas cannot hoist the products (an earlier version with loop-invariant operands was strength-reduced to
// IADD3 / IADD3.X pairs and reported an "IMAD.WIDE" rate that was really the 64-bit add rate).  64 IMAD.WIDE.U32 + 16
// ALU instructions per round; verified in SASS (tools/sass_mix.py).
__global__ void __launch_bounds__(256) k_bench_mad_wide(uint64_t* out, int iters, uint32_t seed) {
    uint32_t x[8], y[8];
    uint64_t t[8];
#pragma unroll
    for (int i = 0; i < 8; i++) { x[i] = seed * (i + 3) + threadIdx.x; y[i] = seed * (i + 11) + blockIdx.x * 7 + threadIdx.x * 13; t[i] = i; }
#pragma unroll 1
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int i = 0; i < 8; i++) {
#pragma unroll
            for (int j = 0; j < 8; j++) t[(i + j) & 7] += (uint64_t)x[i] * y[j];
        }
#pragma unroll
        for (int i = 0; i < 8; i++) { x[i] ^= (uint32_t)t[i]; y[i] += (uint32_t)(t[i] >> 32); }
    }
    uint64_t r = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) r ^= t[i];
    out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = r;
}
__global__ void __launch_bounds__(256) k_bench_mad_carry(uint32_t* out, int iters, uint32_t seed) {
    // the row primitive of fq_mul: 8-limb lo/hi carry chains, two independent accumulators
    uint32_t e[8], o[8];
#pragma unroll
    for (int i = 0; i < 8; i++) { e[i] = seed + i + threadIdx.x; o[i] = seed * 7 + i + blockIdx.x; }
    uint32_t b = seed ^ threadIdx.x;
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int u = 0; u < 4; u++) {
            row_mad(e, o[0], o[2], o[4], o[6], b);
            row_mad(o, e[1], e[3], e[5], e[7], b);
        }
    }
    uint32_t r = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) r ^= e[i] ^ o[i];
    out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = r;
}
template <int PORTABLE>
__global__ void __launch_bounds__(256) k_bench_fq_mul(uint32_t* out, int iters, uint32_t seed) {
    // two independent multiplication chains per thread
    Fq a = fq_one(), b = fq_r2();
    a.l[0] ^= threadIdx.x; b.l[0] ^= blockIdx.x + seed;
    a.l[7] &= 0x0fffffffu; b.l[7] &= 0x0fffffffu;
    Fq c = b, d = a;
    for (int i = 0; i < iters; i++) {
        if (PORTABLE) { a = fq_mul_portable(a, b); c = fq_mul_portable(c, d); }
        else { a = fq_mul(a, b); c = fq_mul(c, d); }
    }
    uint32_t r = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) r ^= a.l[i] ^ c.l[i];
    out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = r;
}


int launch_codec_decode(const uint32_t* in, uint32_t* out, size_t n_fq, int* flags, cudaStream_t s) {
    k_codec_decode<<<(unsigned)((n_fq + 255) / 256), 256, 0, s>>>(in, out, n_fq, flags);
    return (int)cudaGetLastError();
}
int launch_codec_encode(const uint32_t* in, uint32_t* out, size_t n_fq, cudaStream_t s) {
    k_codec_encode<<<(unsigned)((n_fq + 255) / 256), 256, 0, s>>>(in, out, n_fq);
    return (int)cudaGetLastError();
}
int launch_verify_outcome(const uint32_t* proofs, const RaggedProof* pt, size_t count, const uint32_t* z, const uint32_t* pair, const uint32_t* fin,
                          bool enc_finals, int* results, uint32_t* final_A, uint32_t* final_B, uint32_t* final_Z, cudaStream_t s) {
    k_verify_outcome<<<(unsigned)((count * 32 + 127) / 128), 128, 0, s>>>(proofs, pt, count, z, pair, fin, enc_finals ? 1 : 0, results, final_A,
                                                                          final_B, final_Z);
    return (int)cudaGetLastError();
}
int launch_test_fq_op(int op, const uint32_t* a, const uint32_t* b, uint32_t* out, size_t count, cudaStream_t s) {
    k_test_fq_op<<<(unsigned)((count + 127) / 128), 128, 0, s>>>(op, a, b, out, count);
    return (int)cudaGetLastError();
}
int launch_test_fq12_op(int op, const uint32_t* a, const uint32_t* b, uint32_t* out, size_t count, cudaStream_t s) {
    k_test_fq12_op<<<(unsigned)((count + 31) / 32), 32, 0, s>>>(op, a, b, out, count);
    return (int)cudaGetLastError();
}
int launch_microbench(int which, int blocks, int threads, void* out, int iters, uint32_t seed, double* ops_per_thread, cudaStream_t s) {
    switch (which) {
        case 0: k_bench_mad_lo<<<blocks, threads, 0, s>>>((uint32_t*)out, iters, seed); *ops_per_thread = 64.0 * iters; break;
        case 1: k_bench_mad_wide<<<blocks, threads, 0, s>>>((uint64_t*)out, iters, seed); *ops_per_thread = 64.0 * iters; break;
        case 2: k_bench_mad_carry<<<blocks, threads, 0, s>>>((uint32_t*)out, iters, seed); *ops_per_thread = 64.0 * iters; break;
        case 3: k_bench_fq_mul<0><<<blocks, threads, 0, s>>>((uint32_t*)out, iters, seed); *ops_per_thread = 2.0 * iters; break;
        case 4: k_bench_fq_mul<1><<<blocks, threads, 0, s>>>((uint32_t*)out, iters, seed); *ops_per_thread = 2.0 * iters; break;
        default: return -1;
    }
    return (int)cudaGetLastError();
}

}  // namespace sipp

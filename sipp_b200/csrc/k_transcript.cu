// k_transcript.cu -- the Fiat-Shamir transcript on the device, one hash chain per SIPP instance (batched proving,
// BASELINE config "4096 independent n=128 instances").
//
// A single proof keeps its transcript on the host (transcript.cc): the chain is strictly sequential and a CPU core runs
// it faster than a GPU thread.  A batch of independent instances has one independent chain per instance, so the chains
// run side by side here and whole instances stay resident in HBM: no challenge ever crosses PCIe.
//
// Mirrors /root/reference/src/transcript_native.rs:14-77 (`Transcript<GoldilocksField>`):
//   append      state <- hash_n_to_hash_no_pad(state || msg)   :25-30  (overwrite-mode sponge, rate 8, width 12)
//   append_g1 / append_g2 / append_fq12                        :32-54  (8 little-endian u32 limbs per Fq, MyFq12 order)
//   get_challenge                                              :56-65  (zero-stripped u32 digits of the digest, mod r)
// followed by what the prover does with the challenge: x^-1 (prover_native.rs:58) and the GLV / GLS recoding the fold
// kernel consumes (glv_core.h).  The permutation is the textbook Poseidon (30 rounds of constants, S-box, MDS): the same
// function as the host's sparse-matrix formulation (tests compare the two), computed by 16 lanes per instance, one lane per
// state element.
#include <cuda_runtime.h>
#include <stdint.h>

#define SIPP_GLV_CONST static __device__ const
#include "glv_consts.h"
#include "glv_core.h"
#include "launch.h"
#include "poseidon_rc.h"

namespace sipp {

namespace {

__constant__ uint64_t c_rc[360];
bool g_rc_loaded[64] = {false};

#define GL_EPS 0xFFFFFFFFull
#define GL_P 0xFFFFFFFF00000001ull

__device__ __forceinline__ uint64_t gl_add(uint64_t a, uint64_t b) {  // any u64 representatives
    uint64_t r = a + b;
    if (r < a) {  // wrapped: 2^64 = EPS (mod p)
        uint64_t t = r + GL_EPS;
        r = t < r ? t + GL_EPS : t;
    }
    return r;
}
// x = hi * 2^64 + lo  ->  representative in [0, 2^64)
__device__ __forceinline__ uint64_t gl_reduce128(uint64_t lo, uint64_t hi) {
    uint64_t hh = hi >> 32, hl = hi & GL_EPS;
    uint64_t t = lo - hh;  // 2^96 = -1
    if (lo < hh) t -= GL_EPS;
    uint64_t m = hl * GL_EPS;  // 2^64 = 2^32 - 1
    uint64_t r = t + m;
    if (r < m) r += GL_EPS;
    return r;
}
__device__ __forceinline__ uint64_t gl_mul(uint64_t a, uint64_t b) { return gl_reduce128(a * b, __umul64hi(a, b)); }
__device__ __forceinline__ uint64_t gl_pow7(uint64_t x) {
    uint64_t x2 = gl_mul(x, x), x3 = gl_mul(x2, x), x4 = gl_mul(x2, x2);
    return gl_mul(x3, x4);
}
__device__ __forceinline__ uint64_t gl_canon(uint64_t a) { return a >= GL_P ? a - GL_P : a; }

// ---- one permutation on a group of 16 lanes: lane l < 12 holds state element l (lanes 12..15 shadow lanes 0..3 and are
// ignored).  Per round every lane adds its constant, raises to the 7th power (all lanes in a full round, lane 0 in a partial
// round) and gathers its MDS row with 24 shuffles: the dependent chain of a permutation is ~30 x (S-box + 24 multiply-adds)
// instead of 30 x 12 x that on one thread, which is what the strictly sequential absorb chain of an instance needs.
// rc: the 360 round constants in shared memory.
__device__ __forceinline__ uint64_t poseidon_lanes(uint64_t s, int l, const uint64_t* rc) {
    const uint32_t C[12] = {17, 15, 41, 16, 2, 28, 13, 13, 39, 18, 34, 20};
    const int lc = l < 12 ? l : l - 12;
#pragma unroll 1
    for (int rnd = 0; rnd < 30; rnd++) {
        s = gl_add(s, rc[12 * rnd + lc]);
        if (rnd < 4 || rnd >= 26 || lc == 0) s = gl_pow7(s);
        const uint32_t lo = (uint32_t)s, hi = (uint32_t)(s >> 32);
        uint64_t al = 0, ah = 0;
        int src = lc;
#pragma unroll
        for (int i = 0; i < 12; i++) {
            const uint32_t vlo = __shfl_sync(0xffffffffu, lo, src, 16), vhi = __shfl_sync(0xffffffffu, hi, src, 16);
            al += (uint64_t)vlo * C[i];
            ah += (uint64_t)vhi * C[i];
            src = src == 11 ? 0 : src + 1;
        }
        if (lc == 0) { al += (uint64_t)lo * 8; ah += (uint64_t)hi * 8; }
        // value = al + ah 2^32 < 2^75
        const uint64_t lw = al + (ah << 32);
        const uint64_t hw = (ah >> 32) + (lw < al ? 1 : 0);  // < 2^11
        const uint64_t m = hw * GL_EPS;
        uint64_t x = lw + m;
        if (x < m) x += GL_EPS;
        s = x;
    }
    return gl_canon(s);
}

// state <- hash_n_to_hash_no_pad(state || msg) on a lane group: lanes 0..3 hold the state in `s` on entry and on return;
// msg = n u32-valued field elements read through get(i) (every lane calls it with its own index)
template <class Get>
__device__ __forceinline__ uint64_t tr_append_lanes(uint64_t s, int l, const uint64_t* rc, int n, Get get) {
    const int lc = l < 12 ? l : l - 12;
    const int first = n < 4 ? n : 4;
    if (lc >= 4) s = (lc < 4 + first) ? get(lc - 4) : 0;
    s = poseidon_lanes(s, l, rc);
    for (int off = first; off < n; off += 8) {
        const int len = n - off < 8 ? n - off : 8;
        if (lc < len) s = get(off + lc);
        s = poseidon_lanes(s, l, rc);
    }
    return s;
}

// f: 96 canonical u32 words in the boundary (ark nested) order; order 0 = MyFq12 w-basis, 1 = nested
__device__ __forceinline__ uint64_t tr_append_fq12_lanes(uint64_t s, int l, const uint64_t* rc, const uint32_t* f, int order) {
    return tr_append_lanes(s, l, rc, 96, [&](int i) -> uint64_t {
        if (order == 1) return f[i];
        int c = i >> 3, w = i & 7;          // coefficient c of MyFq12.coeffs, limb w
        int g = c < 6 ? c : c - 6;          // Fq2 coefficient of w^g; c >= 6 selects its c1
        int slot = (g & 1) * 3 + (g >> 1);
        return f[16 * slot + (c < 6 ? 0 : 8) + w];
    });
}

// the lattice tables of the device recoding (glv_consts.h as __device__ constants)
__device__ __forceinline__ glv::Tables device_glv_tables() {
    return glv::Tables{&SIPP_GLV_G1_BASIS[0][0][0], &SIPP_GLV_G1_RECIP[0][0], SIPP_GLV_G1_RECIP_SIGN,
                       &SIPP_GLS_G2_BASIS[0][0][0], &SIPP_GLS_G2_RECIP[0][0], SIPP_GLS_G2_RECIP_SIGN};
}

__device__ __forceinline__ void load_rc_shared(uint64_t* rc) {
    for (int i = threadIdx.x; i < 360; i += blockDim.x) rc[i] = c_rc[i];
    __syncthreads();
}

}  // namespace

// register n pairs (prover_native.rs:36-39) on a lane group, from Transcript::new (transcript_native.rs:19-23)
__device__ __forceinline__ uint64_t absorb_pairs_lanes(const uint32_t* a, const uint32_t* b, size_t n, int l, const uint64_t* rc) {
    uint64_t s = 0;
    for (size_t i = 0; i < n; i++) {
        const uint32_t* pa = a + 16 * i;
        const uint32_t* pb = b + 32 * i;
        s = tr_append_lanes(s, l, rc, 16, [&](int k) -> uint64_t { return pa[k]; });  // append_g1  :42-46
        s = tr_append_lanes(s, l, rc, 32, [&](int k) -> uint64_t { return pb[k]; });  // append_g2  :48-54
    }
    return s;
}

#define SIPP_TR_THREADS 32  // two instances per block: the chains are latency-bound, spread them over the SMs

// 16 lanes per instance: register A and B (prover_native.rs:36-39), 8 permutations per pair
__global__ void __launch_bounds__(SIPP_TR_THREADS) k_tr_absorb_pairs(const uint32_t* __restrict__ bytesA, const uint32_t* __restrict__ bytesB, size_t n, size_t count,
                                                                     uint64_t* __restrict__ states) {
    __shared__ uint64_t rc[360];
    load_rc_shared(rc);
    const int l = threadIdx.x & 15;
    size_t inst = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 4;
    const bool have = inst < count;
    if (!have) inst = count - 1;  // shadow: the shuffles need every lane of the warp
    const uint64_t s = absorb_pairs_lanes(bytesA + inst * n * 16, bytesB + inst * n * 32, n, l, rc);
    if (have && l < 4) states[4 * inst + l] = s;
}

// ragged batch: instance k absorbs pairs [tab[k].base, tab[k].base + 2 tab[k].h) (round 1's table: n_k = 2h).  The chain of an
// instance is 8 n_k permutations, so the longest instance bounds the launch.
__global__ void __launch_bounds__(SIPP_TR_THREADS) k_tr_absorb_pairs_ragged(const uint32_t* __restrict__ bytesA, const uint32_t* __restrict__ bytesB,
                                                                            const RaggedInst* __restrict__ tab, unsigned act, uint64_t* __restrict__ states) {
    __shared__ uint64_t rc[360];
    load_rc_shared(rc);
    const int l = threadIdx.x & 15;
    size_t inst = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 4;
    const bool have = inst < act;
    if (!have) inst = act - 1;
    const RaggedInst r = tab[inst];
    const uint64_t s = absorb_pairs_lanes(bytesA + (size_t)r.base * 16, bytesB + (size_t)r.base * 32, 2 * (size_t)r.h, l, rc);
    if (have && l < 4) states[4 * inst + l] = s;
}

// 16 lanes per instance absorb Z (first round only), Z_L, Z_R and derive the digest; lane 0 then turns it into the challenge,
// inverts it and recodes it.  proofs: [count][np][96 words] boundary bytes; slots index the Fq12 inside an instance's proof
// (slot_z < 0: skip).  flags[0] |= 1 on a zero challenge (x.inverse().unwrap() panics in the reference), |= 2 on a recoding
// failure.
// the round of instance `inst` (pf: its proof) on a lane group
__device__ __forceinline__ void tr_round_lanes(uint64_t* __restrict__ states, const uint32_t* pf, int slot_z, int slot_l, int slot_r, int order, size_t inst,
                                               bool have, int l, const uint64_t* rc, FoldPlan* __restrict__ plans, uint64_t* __restrict__ challenges,
                                               int* __restrict__ flags) {
    uint64_t s = states[4 * inst + (l & 3)];
    if (slot_z >= 0) s = tr_append_fq12_lanes(s, l, rc, pf + (size_t)slot_z * 96, order);  // prover_native.rs:42-43
    s = tr_append_fq12_lanes(s, l, rc, pf + (size_t)slot_l * 96, order);                    // :52-53
    s = tr_append_fq12_lanes(s, l, rc, pf + (size_t)slot_r * 96, order);                    // :54-55
    if (have && l < 4) states[4 * inst + l] = s;
    // get_challenge (&self: the state is not advanced)  transcript_native.rs:56-65
    uint64_t d = poseidon_lanes(l < 4 ? s : 0, l, rc);
    uint64_t dg[4];
#pragma unroll
    for (int k = 0; k < 4; k++) dg[k] = __shfl_sync(0xffffffffu, d, k, 16);
    if (!have || l != 0) return;
    uint32_t digits[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    int nd = 0;
    for (int k = 0; k < 4; k++) {  // to_u32_digits strips high zero digits (0 -> no digit at all)
        uint64_t t = dg[k];
        while (t) {
            digits[nd++] = (uint32_t)t;
            t >>= 32;
        }
    }
    uint64_t v[4];
    for (int j = 0; j < 4; j++) v[j] = (uint64_t)digits[2 * j] | ((uint64_t)digits[2 * j + 1] << 32);
    const uint64_t RM[4] = {0x43e1f593f0000001ull, 0x2833e84879b97091ull, 0xb85045b68181585dull, 0x30644e72e131a029ull};
    for (int it = 0; it < 6 && glv::fr_geq(v, RM); it++) {  // v < 2^256 < 6r
        uint64_t borrow = 0;
        for (int i = 0; i < 4; i++) {
            unsigned __int128 t = (unsigned __int128)v[i] - RM[i] - borrow;
            v[i] = (uint64_t)t;
            borrow = (uint64_t)(t >> 64) & 1;
        }
    }
    uint64_t vi[4] = {0, 0, 0, 0};
    int rc_inv = glv::fr_inverse_binary(v, vi);                                    // prover_native.rs:58
    if (challenges) {
        for (int i = 0; i < 4; i++) { challenges[8 * inst + i] = v[i]; challenges[8 * inst + 4 + i] = vi[i]; }
    }
    FoldPlan plan;
    for (int i = 0; i < (int)(sizeof(FoldPlan) / 4); i++) ((uint32_t*)&plan)[i] = 0;
    if (rc_inv) {
        atomicOr(flags, 1);
    } else {
        if (glv::plan_build(v, vi, device_glv_tables(), &plan)) atomicOr(flags, 2);
    }
    plans[inst] = plan;
}
__global__ void __launch_bounds__(SIPP_TR_THREADS) k_tr_round(uint64_t* __restrict__ states, const uint32_t* __restrict__ proofs, size_t np, int slot_z, int slot_l,
                                                              int slot_r, int order, size_t count, FoldPlan* __restrict__ plans, uint64_t* __restrict__ challenges,
                                                              int* __restrict__ flags) {
    __shared__ uint64_t rc[360];
    load_rc_shared(rc);
    const int l = threadIdx.x & 15;
    size_t inst = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 4;
    const bool have = inst < count;
    if (!have) inst = count - 1;
    tr_round_lanes(states, proofs + inst * np * 96, slot_z, slot_l, slot_r, order, inst, have, l, rc, plans, challenges, flags);
}

// ragged batch, round `round` >= 1 of the active instances k < act: instance k's proof is pt[k] (its own np), its slots those of
// batch.cu (Z at np - 1, absorbed in round 1 only; Z_L at np - 2 round, Z_R at np - 1 - 2 round).  challenges (or NULL: the prover)
// receive x || x^-1 of every instance, for the verifier's GT updates.
__global__ void __launch_bounds__(SIPP_TR_THREADS) k_tr_round_ragged(uint64_t* __restrict__ states, const uint32_t* __restrict__ proofs,
                                                                     const RaggedProof* __restrict__ pt, int round, int order, unsigned act,
                                                                     FoldPlan* __restrict__ plans, uint64_t* __restrict__ challenges,
                                                                     int* __restrict__ flags) {
    __shared__ uint64_t rc[360];
    load_rc_shared(rc);
    const int l = threadIdx.x & 15;
    size_t inst = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 4;
    const bool have = inst < act;
    if (!have) inst = act - 1;
    const RaggedProof p = pt[inst];
    const int np = (int)p.np;
    tr_round_lanes(states, proofs + p.first * 96, round == 1 ? np - 1 : -1, np - 2 * round, np - 1 - 2 * round, order, inst, have, l, rc, plans, challenges,
                   flags);
}

// test hook: the recoding k_tr_round runs, on given pairs (xs, xinvs: 4 u64 each), one thread per pair; fails counts the pairs
// plan_build refused
__global__ void __launch_bounds__(64) k_test_plan_build(const uint64_t* __restrict__ xs, const uint64_t* __restrict__ xinvs, size_t count,
                                                         FoldPlan* __restrict__ plans, int* __restrict__ fails) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    uint64_t kx[4], ki[4];
    for (int w = 0; w < 4; w++) { kx[w] = xs[4 * i + w]; ki[w] = xinvs[4 * i + w]; }
    FoldPlan plan;
    for (int w = 0; w < (int)(sizeof(FoldPlan) / 4); w++) ((uint32_t*)&plan)[w] = 0;
    if (glv::plan_build(kx, ki, device_glv_tables(), &plan)) atomicAdd(fails, 1);
    plans[i] = plan;
}

// test hook: `count` independent permutations, 16 lanes each
__global__ void __launch_bounds__(SIPP_TR_THREADS) k_test_poseidon(uint64_t* __restrict__ states, size_t count) {
    __shared__ uint64_t rc[360];
    load_rc_shared(rc);
    const int l = threadIdx.x & 15;
    size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 4;
    const bool have = i < count;
    if (!have) i = count - 1;
    uint64_t s = poseidon_lanes(states[12 * i + (l < 12 ? l : l - 12)], l, rc);
    if (have && l < 12) states[12 * i + l] = s;
}

static int load_rc() {
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev >= 0 && dev < 64 && g_rc_loaded[dev]) return 0;
    cudaError_t e = cudaMemcpyToSymbol(c_rc, SIPP_POSEIDON_RC, sizeof(uint64_t) * 360);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();  // once per device: the kernels run on a non-blocking stream
    if (e != cudaSuccess) return (int)e;
    if (dev >= 0 && dev < 64) g_rc_loaded[dev] = true;
    return 0;
}

int launch_tr_absorb_pairs(const uint32_t* bytesA, const uint32_t* bytesB, size_t n, size_t count, uint64_t* states, cudaStream_t s) {
    int e = load_rc();
    if (e) return e;
    k_tr_absorb_pairs<<<(unsigned)((count * 16 + SIPP_TR_THREADS - 1) / SIPP_TR_THREADS), SIPP_TR_THREADS, 0, s>>>(bytesA, bytesB, n, count, states);
    return (int)cudaGetLastError();
}
int launch_tr_round(uint64_t* states, const uint32_t* proofs, size_t np, int slot_z, int slot_l, int slot_r, int order, size_t count, FoldPlan* plans,
                    uint64_t* challenges, int* flags, cudaStream_t s) {
    int e = load_rc();
    if (e) return e;
    k_tr_round<<<(unsigned)((count * 16 + SIPP_TR_THREADS - 1) / SIPP_TR_THREADS), SIPP_TR_THREADS, 0, s>>>(states, proofs, np, slot_z, slot_l, slot_r, order, count, plans, challenges, flags);
    return (int)cudaGetLastError();
}
int launch_tr_absorb_pairs_ragged(const uint32_t* bytesA, const uint32_t* bytesB, const RaggedInst* tab, unsigned act, uint64_t* states, cudaStream_t s) {
    int e = load_rc();
    if (e) return e;
    k_tr_absorb_pairs_ragged<<<(unsigned)(((size_t)act * 16 + SIPP_TR_THREADS - 1) / SIPP_TR_THREADS), SIPP_TR_THREADS, 0, s>>>(bytesA, bytesB, tab, act, states);
    return (int)cudaGetLastError();
}
int launch_tr_round_ragged(uint64_t* states, const uint32_t* proofs, const RaggedProof* pt, int round, int order, unsigned act, FoldPlan* plans,
                           uint64_t* challenges, int* flags, cudaStream_t s) {
    int e = load_rc();
    if (e) return e;
    k_tr_round_ragged<<<(unsigned)(((size_t)act * 16 + SIPP_TR_THREADS - 1) / SIPP_TR_THREADS), SIPP_TR_THREADS, 0, s>>>(states, proofs, pt, round, order, act, plans,
                                                                                                                        challenges, flags);
    return (int)cudaGetLastError();
}
int launch_test_plan_build(const uint64_t* xs, const uint64_t* xinvs, size_t count, FoldPlan* plans, int* fails, cudaStream_t s) {
    k_test_plan_build<<<(unsigned)((count + 63) / 64), 64, 0, s>>>(xs, xinvs, count, plans, fails);
    return (int)cudaGetLastError();
}
int launch_test_poseidon(uint64_t* states, size_t count, cudaStream_t s) {
    int e = load_rc();
    if (e) return e;
    k_test_poseidon<<<(unsigned)((count * 16 + SIPP_TR_THREADS - 1) / SIPP_TR_THREADS), SIPP_TR_THREADS, 0, s>>>(states, count);
    return (int)cudaGetLastError();
}

}  // namespace sipp

// k_msm.cu -- batched multi-scalar multiplications in G1 and G2 (host driver msm.cu; algorithm and shared code: msm.cuh).
//
//   k_msm_recode    one thread per point: scalar check, GLV / GLS split, the term table (-1)^neg endo^j(P), then per term either its
//                   NAF masks (Straus segments) or one sort entry per window (Pippenger segments: key = bucket, value = term << 1 | sign;
//                   a zero digit gets the key `nbuckets`, which sorts behind every bucket and is never read)
//   (CUB radix sort of the entries by key)
//   k_msm_chunks    one thread per chunk of SIPP_MSM_CHUNK sorted entries: mixed additions of each run of equal keys; a run that is a whole
//                   bucket is stored there, the runs cut by the chunk's ends go to its first / last partial
//   k_msm_buckets   one thread per bucket whose run crosses chunks: binary search of the run, sum of the partials of its chunks; a run
//                   over more than SIPP_MSM_LONG_SPAN chunks is queued for k_msm_long_buckets (SIPP_MSM_LONG_PARTS blocks per such
//                   bucket) and k_msm_long_finish (one block per such bucket)
//   k_msm_windows   one block per (window, part of its buckets): running sums per thread, block tree sum -> one partial
//   k_msm_finish    one thread per Pippenger segment: the partials of every window, Horner over the windows, affine
//   k_msm_straus    one thread per Straus segment: shared doublings over the NAF digits of all its terms, affine
#define SIPP_CURVE_FQ2_CALLS 1
#define SIPP_FQ_CALLS 1
#define SIPP_GLV_CONST static __device__ const
#include <cub/device/device_radix_sort.cuh>

#include "device_common.cuh"
#include "glv_consts.h"
#include "msm.cuh"

namespace sipp {

namespace {

__device__ __forceinline__ glv::Tables msm_glv_tables() {
    return glv::Tables{&SIPP_GLV_G1_BASIS[0][0][0], &SIPP_GLV_G1_RECIP[0][0], SIPP_GLV_G1_RECIP_SIGN,
                       &SIPP_GLS_G2_BASIS[0][0][0], &SIPP_GLS_G2_RECIP[0][0], SIPP_GLS_G2_RECIP_SIGN};
}

template <class F>
__device__ __forceinline__ Affine<F> load_point(const uint32_t* p, size_t i);
template <>
__device__ __forceinline__ G1A load_point<Fq>(const uint32_t* p, size_t i) { return load_g1(p, i); }
template <>
__device__ __forceinline__ G2A load_point<Fq2>(const uint32_t* p, size_t i) { return load_g2(p, i); }
template <class F>
__device__ __forceinline__ void store_point(uint32_t* p, size_t i, const Affine<F>& v);
template <>
__device__ __forceinline__ void store_point<Fq>(uint32_t* p, size_t i, const G1A& v) { store_g1(p, i, v); }
template <>
__device__ __forceinline__ void store_point<Fq2>(uint32_t* p, size_t i, const G2A& v) { store_g2(p, i, v); }

}  // namespace

template <class F>
__global__ void __launch_bounds__(128) k_msm_recode(const uint32_t* __restrict__ points, const uint32_t* __restrict__ scalars, uint32_t n,
                                                    const MsmSeg* __restrict__ segs, uint32_t count, Affine<F>* __restrict__ terms,
                                                    FoldComp* __restrict__ naf, uint32_t* __restrict__ keys, uint32_t* __restrict__ vals,
                                                    uint32_t nbuckets, int* __restrict__ flags) {
    constexpr int NC = msm::Group<F>::NC, BITS = msm::Group<F>::BITS;
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const MsmSeg sg = segs[msm::segment_of(segs, count, i)];
    uint32_t k[8];  // word by word: the caller's scalars need only be 4-byte aligned (as in k_bls.cu)
#pragma unroll
    for (int w = 0; w < 8; w++) k[w] = scalars[8 * (size_t)i + w];
    FoldSubScalar sub[NC];
    // flags |= 8: scalar >= r; |= 16: a sub-scalar out of its bound (cannot happen for k < r).  The call then fails: whatever is
    // computed below is never read back.
    const int bad = !msm::scalar_below_r(k) ? 8 : msm::split<F>(k, msm_glv_tables(), sub) ? 16 : 0;
    if (bad) {
        atomicOr(flags, bad);
        for (int j = 0; j < NC; j++) sub[j] = FoldSubScalar{{0, 0, 0}, 0};
    }
    const Affine<F> p = load_point<F>(points, i);
#pragma unroll 1
    for (int j = 0; j < NC; j++) {
        const uint32_t t = i * NC + j;
        terms[t] = msm::term_point(p, j, sub[j].neg);
        if (sg.c == 0) {
            FoldComp fc;
            glv::naf(sub[j].mag, fc.plus, fc.minus);
            fc.neg = 0;
            naf[t] = fc;
        } else {
            const int W = msm::windows(BITS, (int)sg.c);
            const uint32_t nb = 1u << (sg.c - 1);
            const size_t e0 = (size_t)sg.ebase + ((size_t)(i - sg.first) * NC + j) * W;
            msm::signed_digits(sub[j].mag, BITS, (int)sg.c, [&](int w, int d) {
                keys[e0 + w] = d ? sg.bbase + (uint32_t)w * nb + (uint32_t)(d < 0 ? -d : d) - 1 : nbuckets;
                vals[e0 + w] = t << 1 | (d < 0 ? 1u : 0u);
            });
        }
    }
}

template <class F>
__global__ void __launch_bounds__(64) k_msm_chunks(const uint32_t* __restrict__ keys, const uint32_t* __restrict__ vals, uint32_t entries,
                                                   uint32_t nbuckets, const Affine<F>* __restrict__ terms, Jac<F>* __restrict__ buckets,
                                                   Jac<F>* __restrict__ first, Jac<F>* __restrict__ last) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= (entries + SIPP_MSM_CHUNK - 1) / SIPP_MSM_CHUNK) return;
    msm::chunk_sums(keys, vals, entries, nbuckets, k, SIPP_MSM_CHUNK, terms, buckets, first, last);
}
template <class F>
__global__ void __launch_bounds__(64) k_msm_buckets(const uint32_t* __restrict__ keys, uint32_t entries, uint32_t nbuckets, const Jac<F>* __restrict__ first,
                                                    const Jac<F>* __restrict__ last, Jac<F>* __restrict__ buckets, uint32_t* __restrict__ long_list) {
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nbuckets) return;
    if (!msm::bucket_combine(keys, entries, b, SIPP_MSM_CHUNK, SIPP_MSM_LONG_SPAN, first, last, buckets))
        long_list[1 + atomicAdd(long_list, 1u)] = b;  // long_list[0]: the count
}

// the buckets that cross more than SIPP_MSM_LONG_SPAN chunks (an unweighted sum, k_i = 1, puts every term in one bucket): block (x, y)
// sums part y of the chunk partials of queued bucket x (strided over its threads, then a shared-memory tree) into parts[x][y];
// k_msm_long_finish adds the SIPP_MSM_LONG_PARTS parts of each.  Blocks past the number of queued buckets return at once.
#define SIPP_MSM_LONG_THREADS 64
template <class F>
__device__ __forceinline__ Jac<F> block_tree_sum(Jac<F>* sh, Jac<F> acc, int tid) {
    for (int s = SIPP_MSM_LONG_THREADS >> 1; s > 0; s >>= 1) {
        __syncthreads();
        if (tid >= s && tid < 2 * s) sh[tid] = acc;
        __syncthreads();
        if (tid < s) acc = jac_add(acc, sh[tid + s]);
    }
    return acc;
}
template <class F>
__global__ void __launch_bounds__(SIPP_MSM_LONG_THREADS) k_msm_long_buckets(const uint32_t* __restrict__ keys, uint32_t entries,
                                                                            const Jac<F>* __restrict__ first, const Jac<F>* __restrict__ last,
                                                                            Jac<F>* __restrict__ parts, const uint32_t* __restrict__ long_list) {
    __shared__ Jac<F> sh[SIPP_MSM_LONG_THREADS];
    if (blockIdx.x >= long_list[0]) return;
    const uint32_t b = long_list[1 + blockIdx.x];
    const uint32_t lo = msm::lower_bound(keys, entries, b), hi = msm::lower_bound(keys, entries, b + 1);
    const uint32_t kl = lo / SIPP_MSM_CHUNK, kh = (hi - 1) / SIPP_MSM_CHUNK;
    const uint32_t per = (kh - kl + SIPP_MSM_LONG_PARTS - 1) / SIPP_MSM_LONG_PARTS;  // chunk partials kl + 1 .. kh, `per` to a part
    const uint32_t k0 = kl + 1 + blockIdx.y * per, k1 = k0 + per < kh + 1 ? k0 + per : kh + 1;
    const int tid = threadIdx.x;
    Jac<F> acc = blockIdx.y == 0 && tid == 0 ? last[kl] : jac_identity<F>();
    for (uint32_t k = k0 + tid; k < k1; k += SIPP_MSM_LONG_THREADS) acc = jac_add(acc, first[k]);
    acc = block_tree_sum(sh, acc, tid);
    if (tid == 0) parts[(size_t)blockIdx.x * SIPP_MSM_LONG_PARTS + blockIdx.y] = acc;
}
template <class F>
__global__ void __launch_bounds__(SIPP_MSM_LONG_THREADS) k_msm_long_finish(const Jac<F>* __restrict__ parts, Jac<F>* __restrict__ buckets,
                                                                           const uint32_t* __restrict__ long_list) {
    __shared__ Jac<F> sh[SIPP_MSM_LONG_THREADS];
    if (blockIdx.x >= long_list[0]) return;
    const int tid = threadIdx.x;
    Jac<F> acc = jac_identity<F>();
    for (int q = tid; q < SIPP_MSM_LONG_PARTS; q += SIPP_MSM_LONG_THREADS) acc = jac_add(acc, parts[(size_t)blockIdx.x * SIPP_MSM_LONG_PARTS + q]);
    acc = block_tree_sum(sh, acc, tid);
    if (tid == 0) buckets[long_list[1 + blockIdx.x]] = acc;
}

#define SIPP_MSM_WIN_THREADS 64
template <class F>
__global__ void __launch_bounds__(SIPP_MSM_WIN_THREADS) k_msm_windows(const Jac<F>* __restrict__ buckets, const MsmWin* __restrict__ wins,
                                                                      Jac<F>* __restrict__ parts) {
    __shared__ Jac<F> sh[SIPP_MSM_WIN_THREADS];
    const MsmWin wn = wins[blockIdx.x];
    const int tid = threadIdx.x;
    const uint32_t chunk = (wn.count + SIPP_MSM_WIN_THREADS - 1) / SIPP_MSM_WIN_THREADS;
    uint32_t lo = wn.lo + tid * chunk, hi = lo + chunk;
    if (hi > wn.lo + wn.count) hi = wn.lo + wn.count;
    Jac<F> acc = lo < hi ? msm::window_part(buckets + wn.bucket0, lo, hi) : jac_identity<F>();
    for (int s = SIPP_MSM_WIN_THREADS >> 1; s > 0; s >>= 1) {
        __syncthreads();
        if (tid >= s && tid < 2 * s) sh[tid] = acc;
        __syncthreads();
        if (tid < s) acc = jac_add(acc, sh[tid + s]);
    }
    if (tid == 0) parts[blockIdx.x] = acc;
}

// out[seg] (Montgomery affine) for the Pippenger segments listed in idx
template <class F>
__global__ void __launch_bounds__(64) k_msm_finish(const Jac<F>* __restrict__ parts, const MsmSeg* __restrict__ segs, const uint32_t* __restrict__ idx,
                                                   uint32_t nseg, uint32_t* __restrict__ out) {
    const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nseg) return;
    const uint32_t j = idx[q];
    const MsmSeg sg = segs[j];
    const int c = (int)sg.c, W = msm::windows(msm::Group<F>::BITS, c);
    Jac<F> acc = jac_identity<F>();
    for (int w = W - 1; w >= 0; w--) {
        if (w < W - 1)
            for (int i = 0; i < c; i++) acc = jac_dbl(acc);
        for (uint32_t p = 0; p < sg.parts; p++) acc = jac_add(acc, parts[sg.wbase + (uint32_t)w * sg.parts + p]);
    }
    store_point<F>(out, j, jac_to_affine(acc));
}

template <class F>
__global__ void __launch_bounds__(64) k_msm_straus(const Affine<F>* __restrict__ terms, const FoldComp* __restrict__ naf, const MsmSeg* __restrict__ segs,
                                                   const uint32_t* __restrict__ idx, uint32_t nseg, uint32_t* __restrict__ out) {
    constexpr int NC = msm::Group<F>::NC;
    const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nseg) return;
    const uint32_t j = idx[q];
    const MsmSeg sg = segs[j];
    const size_t t0 = (size_t)sg.first * NC;
    store_point<F>(out, j, jac_to_affine(msm::straus_terms(terms + t0, naf + t0, (size_t)sg.len * NC, msm::Group<F>::BITS + 1)));
}

size_t msm_term_bytes(int group) { return group == 1 ? sizeof(G1A) : sizeof(G2A); }
size_t msm_jac_bytes(int group) { return group == 1 ? sizeof(Jac<Fq>) : sizeof(Jac<Fq2>); }

int launch_msm_recode(int group, const uint32_t* points, const uint32_t* scalars, uint32_t n, const MsmSeg* segs, uint32_t count, void* terms,
                      FoldComp* naf, uint32_t* keys, uint32_t* vals, uint32_t nbuckets, int* flags, cudaStream_t s) {
    const unsigned blocks = (n + 127) / 128;
    if (group == 1) k_msm_recode<Fq><<<blocks, 128, 0, s>>>(points, scalars, n, segs, count, (G1A*)terms, naf, keys, vals, nbuckets, flags);
    else k_msm_recode<Fq2><<<blocks, 128, 0, s>>>(points, scalars, n, segs, count, (G2A*)terms, naf, keys, vals, nbuckets, flags);
    return (int)cudaGetLastError();
}

// temp == NULL: *temp_bytes <- the scratch the sort needs
int msm_sort(void* temp, size_t* temp_bytes, const uint32_t* keys_in, uint32_t* keys_out, const uint32_t* vals_in, uint32_t* vals_out, uint32_t entries,
             int key_bits, cudaStream_t s) {
    return (int)cub::DeviceRadixSort::SortPairs(temp, *temp_bytes, keys_in, keys_out, vals_in, vals_out, (int)entries, 0, key_bits, s);
}

size_t msm_long_list_words(uint32_t entries) { return 1 + ((size_t)entries / SIPP_MSM_CHUNK) / SIPP_MSM_LONG_SPAN + 1; }

int launch_msm_buckets(int group, const uint32_t* keys, const uint32_t* vals, uint32_t entries, uint32_t nbuckets, const void* terms, void* buckets,
                       void* first, void* last, uint32_t* long_list, void* long_parts, cudaStream_t s) {
    const unsigned chunks = (entries + SIPP_MSM_CHUNK - 1) / SIPP_MSM_CHUNK;
    const unsigned cb = (chunks + 63) / 64, bb = (nbuckets + 63) / 64;
    // a bucket crossing more than SIPP_MSM_LONG_SPAN chunks holds more than SIPP_MSM_LONG_SPAN x SIPP_MSM_CHUNK entries: there are
    // fewer such buckets than msm_long_list_words(entries) - 1
    const unsigned lb = (unsigned)(msm_long_list_words(entries) - 1);
    const dim3 lgrid(lb, SIPP_MSM_LONG_PARTS);
    cudaError_t e = cudaMemsetAsync(long_list, 0, sizeof(uint32_t), s);
    if (e != cudaSuccess) return (int)e;
    if (group == 1) {
        k_msm_chunks<Fq><<<cb, 64, 0, s>>>(keys, vals, entries, nbuckets, (const G1A*)terms, (Jac<Fq>*)buckets, (Jac<Fq>*)first, (Jac<Fq>*)last);
        k_msm_buckets<Fq><<<bb, 64, 0, s>>>(keys, entries, nbuckets, (const Jac<Fq>*)first, (const Jac<Fq>*)last, (Jac<Fq>*)buckets, long_list);
        k_msm_long_buckets<Fq><<<lgrid, SIPP_MSM_LONG_THREADS, 0, s>>>(keys, entries, (const Jac<Fq>*)first, (const Jac<Fq>*)last, (Jac<Fq>*)long_parts, long_list);
        k_msm_long_finish<Fq><<<lb, SIPP_MSM_LONG_THREADS, 0, s>>>((const Jac<Fq>*)long_parts, (Jac<Fq>*)buckets, long_list);
    } else {
        k_msm_chunks<Fq2><<<cb, 64, 0, s>>>(keys, vals, entries, nbuckets, (const G2A*)terms, (Jac<Fq2>*)buckets, (Jac<Fq2>*)first, (Jac<Fq2>*)last);
        k_msm_buckets<Fq2><<<bb, 64, 0, s>>>(keys, entries, nbuckets, (const Jac<Fq2>*)first, (const Jac<Fq2>*)last, (Jac<Fq2>*)buckets, long_list);
        k_msm_long_buckets<Fq2><<<lgrid, SIPP_MSM_LONG_THREADS, 0, s>>>(keys, entries, (const Jac<Fq2>*)first, (const Jac<Fq2>*)last,
                                                                        (Jac<Fq2>*)long_parts, long_list);
        k_msm_long_finish<Fq2><<<lb, SIPP_MSM_LONG_THREADS, 0, s>>>((const Jac<Fq2>*)long_parts, (Jac<Fq2>*)buckets, long_list);
    }
    return (int)cudaGetLastError();
}

int launch_msm_windows(int group, const void* buckets, const MsmWin* wins, uint32_t nwins, void* parts, cudaStream_t s) {
    if (group == 1) k_msm_windows<Fq><<<nwins, SIPP_MSM_WIN_THREADS, 0, s>>>((const Jac<Fq>*)buckets, wins, (Jac<Fq>*)parts);
    else k_msm_windows<Fq2><<<nwins, SIPP_MSM_WIN_THREADS, 0, s>>>((const Jac<Fq2>*)buckets, wins, (Jac<Fq2>*)parts);
    return (int)cudaGetLastError();
}

int launch_msm_finish(int group, const void* parts, const MsmSeg* segs, const uint32_t* idx, uint32_t nseg, uint32_t* out, cudaStream_t s) {
    const unsigned blocks = (nseg + 63) / 64;
    if (group == 1) k_msm_finish<Fq><<<blocks, 64, 0, s>>>((const Jac<Fq>*)parts, segs, idx, nseg, out);
    else k_msm_finish<Fq2><<<blocks, 64, 0, s>>>((const Jac<Fq2>*)parts, segs, idx, nseg, out);
    return (int)cudaGetLastError();
}

int launch_msm_straus(int group, const void* terms, const FoldComp* naf, const MsmSeg* segs, const uint32_t* idx, uint32_t nseg, uint32_t* out,
                      cudaStream_t s) {
    const unsigned blocks = (nseg + 63) / 64;
    if (group == 1) k_msm_straus<Fq><<<blocks, 64, 0, s>>>((const G1A*)terms, naf, segs, idx, nseg, out);
    else k_msm_straus<Fq2><<<blocks, 64, 0, s>>>((const G2A*)terms, naf, segs, idx, nseg, out);
    return (int)cudaGetLastError();
}

}  // namespace sipp

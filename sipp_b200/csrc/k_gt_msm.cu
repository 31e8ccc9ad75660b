// k_gt_msm.cu -- batched multi-exponentiations in Fq12 (host driver msm.cu: sipp_gt_msm_batch; bucket logic shared with the MSMs in
// msm.cuh).  Generic Fq12 arithmetic, one element per thread (tower.cuh fq12_mul / fq12_sqr): no Frobenius split, no cyclotomic
// squaring, no inverse, so the results equal square-and-multiply for every Fq12, in GT or not.
//
//   k_gt_msm_decode     one thread per element: scalar < r, 12 coordinates < p, decode into table[i] (w-basis Montgomery, the slot layout
//                       of k_seg_product); an element of a short-path segment copies its scalar for k_gt_msm_pow (k_coop.cu), one of a
//                       Pippenger segment emits one sort entry per window (key = bucket, value = element; unsigned c-bit digits, a zero
//                       digit gets the key `nbuckets`, which sorts behind every bucket and is never read)
//   (CUB radix sort of the entries by key)
//   k_gt_msm_one        every bucket <- 1 (an empty bucket is the identity)
//   k_gt_msm_chunks / _buckets / _long_buckets / _long_finish   the bucket products from the sorted entries, as k_msm_*
//   k_gt_msm_windows    one block per (window, part of its buckets): prod_b S_b^(b + 1) by running products, block tree -> one partial
//   k_gt_msm_finish     one block per Pippenger segment: thread w multiplies the partials of window w, thread 0 runs Horner over the
//                       windows (c squarings each) -> table[first element of the segment]
//   k_gt_msm_encode     the segment products -> boundary bytes
#include "device_common.cuh"
#include "msm.cuh"

namespace sipp {

namespace {

// the group operations of msm.cuh's bucket logic, written multiplicatively: buckets and table entries are Fq12
struct GtOps {
    using T = Fq12;
    using In = Fq12;
    static __device__ __forceinline__ T identity() { return fq12_one(); }
    static __device__ __forceinline__ T add(const T& a, const T& b) { return fq12_mul(a, b); }
    static __device__ __forceinline__ T run(const In* terms, const uint32_t* vals, size_t count) {  // count >= 1
        T acc = terms[vals[0]];
        for (size_t e = 1; e < count; e++) acc = fq12_mul(acc, terms[vals[e]]);
        return acc;
    }
    static __device__ __forceinline__ T mul_small(const T& p, uint32_t v) {  // p^v, v >= 1
        T acc = p;
        for (int i = 30 - __clz(v); i >= 0; i--) {
            acc = fq12_sqr(acc);
            if ((v >> i) & 1u) acc = fq12_mul(acc, p);
        }
        return acc;
    }
};

#define SIPP_GT_MSM_THREADS 64

__device__ __forceinline__ Fq12 block_tree_product(Fq12* sh, Fq12 acc, int tid) {
    for (int s = SIPP_GT_MSM_THREADS >> 1; s > 0; s >>= 1) {
        __syncthreads();
        if (tid >= s && tid < 2 * s) sh[tid] = acc;
        __syncthreads();
        if (tid < s) acc = fq12_mul(acc, sh[tid + s]);
    }
    return acc;
}

}  // namespace

__global__ void __launch_bounds__(128) k_gt_msm_decode(const uint32_t* __restrict__ elems, const uint32_t* __restrict__ scalars, uint32_t n,
                                                       const MsmSeg* __restrict__ segs, uint32_t count, Fq12* __restrict__ table,
                                                       uint32_t* __restrict__ sc, uint32_t* __restrict__ keys, uint32_t* __restrict__ vals,
                                                       uint32_t nbuckets, int* __restrict__ flags) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const MsmSeg sg = segs[msm::segment_of(segs, count, i)];
    uint32_t k[8];  // word by word: the caller's buffers need only be 4-byte aligned
#pragma unroll
    for (int w = 0; w < 8; w++) k[w] = scalars[8 * (size_t)i + w];
    // flags |= 8: scalar >= r; |= 1: a coordinate >= p.  The call then fails: whatever is computed below is never read back.
    int bad = 0;
    if (!msm::scalar_below_r(k)) {
        bad = 8;
#pragma unroll
        for (int w = 0; w < 8; w++) k[w] = 0;
    }
    const uint32_t* e = elems + 96 * (size_t)i;
    const uint32_t P[8] = {SIPP_P0, SIPP_P1, SIPP_P2, SIPP_P3, SIPP_P4, SIPP_P5, SIPP_P6, SIPP_P7};
#pragma unroll 1
    for (int q = 0; q < 12; q++) {
        uint32_t c[8], t[8];
#pragma unroll
        for (int w = 0; w < 8; w++) c[w] = e[8 * q + w];
        if (sub8(t, c, P) == 0) bad |= 1;  // no borrow: value >= p
    }
    if (bad) atomicOr(flags, bad);
    table[i] = fq12_decode(e);
    if (sg.c == 0) {
#pragma unroll
        for (int w = 0; w < 8; w++) sc[8 * (size_t)i + w] = k[w];
        return;
    }
    const int c = (int)sg.c, W = msm::gt_windows(c);
    const uint32_t nb = (1u << c) - 1;
    const size_t e0 = (size_t)sg.ebase + (size_t)(i - sg.first) * W;
#pragma unroll 1
    for (int w = 0; w < W; w++) {
        const uint32_t d = msm::scalar_digit(k, c * w, c);
        keys[e0 + w] = d ? sg.bbase + (uint32_t)w * nb + d - 1 : nbuckets;
        vals[e0 + w] = i;
    }
}

__global__ void __launch_bounds__(128) k_gt_msm_one(Fq12* __restrict__ buckets, uint32_t nbuckets) {
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < nbuckets) buckets[b] = fq12_one();
}

__global__ void __launch_bounds__(SIPP_GT_MSM_THREADS) k_gt_msm_chunks(const uint32_t* __restrict__ keys, const uint32_t* __restrict__ vals, uint32_t entries,
                                                                       uint32_t nbuckets, const Fq12* __restrict__ table, Fq12* __restrict__ buckets,
                                                                       Fq12* __restrict__ first, Fq12* __restrict__ last) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= (entries + SIPP_MSM_CHUNK - 1) / SIPP_MSM_CHUNK) return;
    msm::chunk_sums_of<GtOps>(keys, vals, entries, nbuckets, k, SIPP_MSM_CHUNK, table, buckets, first, last);
}
__global__ void __launch_bounds__(SIPP_GT_MSM_THREADS) k_gt_msm_buckets(const uint32_t* __restrict__ keys, uint32_t entries, uint32_t nbuckets,
                                                                        const Fq12* __restrict__ first, const Fq12* __restrict__ last,
                                                                        Fq12* __restrict__ buckets, uint32_t* __restrict__ long_list) {
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nbuckets) return;
    if (!msm::bucket_combine_of<GtOps>(keys, entries, b, SIPP_MSM_CHUNK, SIPP_MSM_LONG_SPAN, first, last, buckets))
        long_list[1 + atomicAdd(long_list, 1u)] = b;  // long_list[0]: the count
}
// buckets over more than SIPP_MSM_LONG_SPAN chunks (an unweighted product puts every element of a segment in one bucket): as
// k_msm_long_buckets / k_msm_long_finish, SIPP_MSM_LONG_PARTS blocks per queued bucket, then one block adds their parts
__global__ void __launch_bounds__(SIPP_GT_MSM_THREADS) k_gt_msm_long_buckets(const uint32_t* __restrict__ keys, uint32_t entries, const Fq12* __restrict__ first,
                                                                             const Fq12* __restrict__ last, Fq12* __restrict__ parts,
                                                                             const uint32_t* __restrict__ long_list) {
    __shared__ Fq12 sh[SIPP_GT_MSM_THREADS];
    if (blockIdx.x >= long_list[0]) return;
    const uint32_t b = long_list[1 + blockIdx.x];
    const uint32_t lo = msm::lower_bound(keys, entries, b), hi = msm::lower_bound(keys, entries, b + 1);
    const uint32_t kl = lo / SIPP_MSM_CHUNK, kh = (hi - 1) / SIPP_MSM_CHUNK;
    const uint32_t per = (kh - kl + SIPP_MSM_LONG_PARTS - 1) / SIPP_MSM_LONG_PARTS;  // chunk partials kl + 1 .. kh, `per` to a part
    const uint32_t k0 = kl + 1 + blockIdx.y * per, k1 = k0 + per < kh + 1 ? k0 + per : kh + 1;
    const int tid = threadIdx.x;
    Fq12 acc = blockIdx.y == 0 && tid == 0 ? last[kl] : fq12_one();
    for (uint32_t k = k0 + tid; k < k1; k += SIPP_GT_MSM_THREADS) acc = fq12_mul(acc, first[k]);
    acc = block_tree_product(sh, acc, tid);
    if (tid == 0) parts[(size_t)blockIdx.x * SIPP_MSM_LONG_PARTS + blockIdx.y] = acc;
}
__global__ void __launch_bounds__(SIPP_GT_MSM_THREADS) k_gt_msm_long_finish(const Fq12* __restrict__ parts, Fq12* __restrict__ buckets,
                                                                            const uint32_t* __restrict__ long_list) {
    __shared__ Fq12 sh[SIPP_GT_MSM_THREADS];
    if (blockIdx.x >= long_list[0]) return;
    const int tid = threadIdx.x;
    Fq12 acc = fq12_one();
    for (int q = tid; q < SIPP_MSM_LONG_PARTS; q += SIPP_GT_MSM_THREADS) acc = fq12_mul(acc, parts[(size_t)blockIdx.x * SIPP_MSM_LONG_PARTS + q]);
    acc = block_tree_product(sh, acc, tid);
    if (tid == 0) buckets[long_list[1 + blockIdx.x]] = acc;
}

__global__ void __launch_bounds__(SIPP_GT_MSM_THREADS) k_gt_msm_windows(const Fq12* __restrict__ buckets, const MsmWin* __restrict__ wins,
                                                                        Fq12* __restrict__ parts) {
    __shared__ Fq12 sh[SIPP_GT_MSM_THREADS];
    const MsmWin wn = wins[blockIdx.x];
    const int tid = threadIdx.x;
    const uint32_t chunk = (wn.count + SIPP_GT_MSM_THREADS - 1) / SIPP_GT_MSM_THREADS;
    uint32_t lo = wn.lo + tid * chunk, hi = lo + chunk;
    if (hi > wn.lo + wn.count) hi = wn.lo + wn.count;
    Fq12 acc = lo < hi ? msm::window_part_of<GtOps>(buckets + wn.bucket0, lo, hi) : fq12_one();
    acc = block_tree_product(sh, acc, tid);
    if (tid == 0) parts[blockIdx.x] = acc;
}

// block q: Pippenger segment idx[q].  Thread w < W multiplies the partials of window w into the first of them (in place: each block
// owns its segment's partials), then thread 0 runs Horner from the top window and writes table[first element].
#define SIPP_GT_FINISH_THREADS 128
__global__ void __launch_bounds__(SIPP_GT_FINISH_THREADS) k_gt_msm_finish(Fq12* __restrict__ parts, const MsmSeg* __restrict__ segs,
                                                                          const uint32_t* __restrict__ idx, Fq12* __restrict__ table) {
    const MsmSeg sg = segs[idx[blockIdx.x]];
    const int c = (int)sg.c, W = msm::gt_windows(c);
    Fq12* wp = parts + sg.wbase;
    for (int w = threadIdx.x; w < W; w += SIPP_GT_FINISH_THREADS) {
        Fq12 acc = wp[(size_t)w * sg.parts];
        for (uint32_t p = 1; p < sg.parts; p++) acc = fq12_mul(acc, wp[(size_t)w * sg.parts + p]);
        wp[(size_t)w * sg.parts] = acc;
    }
    __syncthreads();
    if (threadIdx.x) return;
    Fq12 acc = wp[(size_t)(W - 1) * sg.parts];
    for (int w = W - 2; w >= 0; w--) {
        for (int i = 0; i < c; i++) acc = fq12_sqr(acc);
        acc = fq12_mul(acc, wp[(size_t)w * sg.parts]);
    }
    table[sg.first] = acc;
}

// out[j] (boundary bytes) <- work[j] (w-basis Montgomery), one thread per ark slot of an Fq12
__global__ void __launch_bounds__(128) k_gt_msm_encode(const uint32_t* __restrict__ work, size_t count, uint32_t* __restrict__ out) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= count * 6) return;
    const size_t j = t / 6;
    const int q = (int)(t % 6);
    const uint32_t* src = work + 96 * j + 16 * fq12_slot_to_w(q);
    Fq2 v;
#pragma unroll
    for (int w = 0; w < 8; w++) {
        v.c0.l[w] = src[w];
        v.c1.l[w] = src[8 + w];
    }
    fq2_encode(out + 96 * j + 16 * q, v);
}

// ------------------------------------------------------------------------------------------------ launch wrappers
int launch_gt_msm_decode(const uint32_t* elems, const uint32_t* scalars, uint32_t n, const MsmSeg* segs, uint32_t count, uint32_t* table, uint32_t* sc,
                         uint32_t* keys, uint32_t* vals, uint32_t nbuckets, int* flags, cudaStream_t s) {
    k_gt_msm_decode<<<(n + 127) / 128, 128, 0, s>>>(elems, scalars, n, segs, count, (Fq12*)table, sc, keys, vals, nbuckets, flags);
    return (int)cudaGetLastError();
}

int launch_gt_msm_buckets(const uint32_t* keys, const uint32_t* vals, uint32_t entries, uint32_t nbuckets, const uint32_t* table, uint32_t* buckets,
                          uint32_t* first, uint32_t* last, uint32_t* long_list, uint32_t* long_parts, cudaStream_t s) {
    const unsigned chunks = (entries + SIPP_MSM_CHUNK - 1) / SIPP_MSM_CHUNK;
    const unsigned cb = (chunks + SIPP_GT_MSM_THREADS - 1) / SIPP_GT_MSM_THREADS, bb = (nbuckets + SIPP_GT_MSM_THREADS - 1) / SIPP_GT_MSM_THREADS;
    const unsigned lb = (unsigned)(msm_long_list_words(entries) - 1);  // as launch_msm_buckets
    const dim3 lgrid(lb, SIPP_MSM_LONG_PARTS);
    cudaError_t e = cudaMemsetAsync(long_list, 0, sizeof(uint32_t), s);
    if (e != cudaSuccess) return (int)e;
    Fq12 *bk = (Fq12*)buckets, *fi = (Fq12*)first, *la = (Fq12*)last, *lp = (Fq12*)long_parts;
    k_gt_msm_one<<<(nbuckets + 127) / 128, 128, 0, s>>>(bk, nbuckets);
    k_gt_msm_chunks<<<cb, SIPP_GT_MSM_THREADS, 0, s>>>(keys, vals, entries, nbuckets, (const Fq12*)table, bk, fi, la);
    k_gt_msm_buckets<<<bb, SIPP_GT_MSM_THREADS, 0, s>>>(keys, entries, nbuckets, fi, la, bk, long_list);
    k_gt_msm_long_buckets<<<lgrid, SIPP_GT_MSM_THREADS, 0, s>>>(keys, entries, fi, la, lp, long_list);
    k_gt_msm_long_finish<<<lb, SIPP_GT_MSM_THREADS, 0, s>>>(lp, bk, long_list);
    return (int)cudaGetLastError();
}

int launch_gt_msm_windows(const uint32_t* buckets, const MsmWin* wins, uint32_t nwins, uint32_t* parts, uint32_t nseg, const MsmSeg* segs,
                          const uint32_t* idx, uint32_t* table, cudaStream_t s) {
    k_gt_msm_windows<<<nwins, SIPP_GT_MSM_THREADS, 0, s>>>((const Fq12*)buckets, wins, (Fq12*)parts);
    k_gt_msm_finish<<<nseg, SIPP_GT_FINISH_THREADS, 0, s>>>((Fq12*)parts, segs, idx, (Fq12*)table);
    return (int)cudaGetLastError();
}

int launch_gt_msm_encode(const uint32_t* work, size_t count, uint32_t* out, cudaStream_t s) {
    k_gt_msm_encode<<<(unsigned)((count * 6 + 127) / 128), 128, 0, s>>>(work, count, out);
    return (int)cudaGetLastError();
}

}  // namespace sipp

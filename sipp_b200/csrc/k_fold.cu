// k_fold.cu -- see kernels overview in device_common.cuh
// Fq2 products are real calls: fully inlined the scalar-multiplication loops are 45-65k SASS instructions, several times the
// instruction cache.
#define SIPP_CURVE_FQ2_CALLS 1
#define SIPP_FQ_CALLS 1
#include "coop.cuh"
#include "device_common.cuh"
#include "fold_map.cuh"
#include "fold_plan.h"
#include "fq2h.cuh"

namespace sipp {

// ------------------------------------------------------------------------------------------------ K4
// Fixed-scalar fold, lane-split over the endomorphism components (fold_plan.h).
//   A_i <- A_i + x A_{i+h}       /root/reference/src/prover_native.rs:60-64
//   B_i <- B_i + x^-1 B_{i+h}    /root/reference/src/prover_native.rs:65-69
// One launch covers both groups.  Blocks [0, g2_blocks) fold 32 G2 elements each: warp j multiplies psi^j(B_{i+h}) by the
// 66-bit sub-scalar k_j (NAF, Jacobian accumulator, mixed additions) -- the digit tests are warp-uniform because a whole
// warp works on the same component; warps 1..3 hand their partial sums to warp 0 through shared memory, which adds them,
// adds B_i and normalises to affine.  The remaining blocks fold 64 G1 elements each the same way with the two GLV
// components (warps 0/1 and 2/3).  Against one thread per element this shortens the dependent chain from 254 doublings
// to 66 (G2) / 128 (G1) at equal total work, which is what the latency-bound rounds (n <= 2^14 per GPU) need.
#define SIPP_FOLD_THREADS 128

template <class F>
__device__ __forceinline__ void store_jac(uint32_t* dst, const Jac<F>& p);
template <>
__device__ __forceinline__ void store_jac<Fq2>(uint32_t* dst, const Jac<Fq2>& p) {
    store_fq2_words(dst, p.x); store_fq2_words(dst + 16, p.y); store_fq2_words(dst + 32, p.z);
}
__device__ __forceinline__ Jac<Fq2> load_jac2(const uint32_t* src) {
    Jac<Fq2> p;
    p.x = load_fq2_words(src); p.y = load_fq2_words(src + 16); p.z = load_fq2_words(src + 32);
    return p;
}
__device__ __forceinline__ void store_fq_words(uint32_t* p, const Fq& v) {
    uint4* q = reinterpret_cast<uint4*>(p);
    q[0] = make_uint4(v.l[0], v.l[1], v.l[2], v.l[3]);
    q[1] = make_uint4(v.l[4], v.l[5], v.l[6], v.l[7]);
}
__device__ __forceinline__ Fq load_fq_words(const uint32_t* p) {
    const uint4* q = reinterpret_cast<const uint4*>(p);
    uint4 a = q[0], b = q[1];
    return Fq{{a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w}};
}
template <>
__device__ __forceinline__ void store_jac<Fq>(uint32_t* dst, const Jac<Fq>& p) {
    store_fq_words(dst, p.x); store_fq_words(dst + 8, p.y); store_fq_words(dst + 16, p.z);
}
__device__ __forceinline__ Jac<Fq> load_jac1(const uint32_t* src) {
    Jac<Fq> p;
    p.x = load_fq_words(src); p.y = load_fq_words(src + 8); p.z = load_fq_words(src + 16);
    return p;
}

// Jacobian point over Fq2H (fq2h.cuh): every lane of a pair moves its halves; same 48-word layout as a Jac<Fq2>
__device__ __forceinline__ void store_jac_h(uint32_t* dst, const Jac<Fq2H>& p) {
    const int o = h_odd() ? 8 : 0;
    store_fq_words(dst + o, p.x.v); store_fq_words(dst + 16 + o, p.y.v); store_fq_words(dst + 32 + o, p.z.v);
}
__device__ __forceinline__ Jac<Fq2H> load_jac_h(const uint32_t* src) {
    const int o = h_odd() ? 8 : 0;
    Jac<Fq2H> p;
    p.x.v = load_fq_words(src + o); p.y.v = load_fq_words(src + 16 + o); p.z.v = load_fq_words(src + 32 + o);
    return p;
}
__device__ __forceinline__ Affine<Fq2H> split_g2(const G2A& q) { return Affine<Fq2H>{h_split(q.x), h_split(q.y)}; }

// ---- G1 on a PAIR of lanes.  An Fq product cannot be split, but the products of a doubling / mixed addition are not all
// dependent: both lanes hold the whole point, each computes one of two independent products per level and the results are
// exchanged with 8 shuffles -- 7 products in 4 levels (doubling), 11 in 6 (mixed addition) instead of 7 / 11 in a row.  The 128
// doublings of a GLV component were the longest chain of the lane-split fold once G2 ran on lane pairs.
__device__ __forceinline__ void pair_mul(const Fq& a_even, const Fq& b_even, const Fq& a_odd, const Fq& b_odd, Fq& r_even, Fq& r_odd) {
    const bool odd = h_odd();
    const Fq mine = fq_mul_call(h_select(odd, a_odd, a_even), h_select(odd, b_odd, b_even));
    const Fq other = h_partner(mine);
    r_even = h_select(odd, other, mine);
    r_odd = h_select(odd, mine, other);
}
__device__ __noinline__ Jac<Fq> jac_dbl_pair(const Jac<Fq>& p) {  // same formulas as jac_dbl (curve.cuh)
    Fq A, B, C, S, Fv, YZ, M, unused;
    pair_mul(p.x, p.x, p.y, p.y, A, B);
    const Fq xb = fq_add(p.x, B);
    pair_mul(B, B, xb, xb, C, S);
    const Fq D = fq_dbl(fq_sub(fq_sub(S, A), C));
    const Fq E = fq_add(fq_dbl(A), A);
    pair_mul(E, E, p.y, p.z, Fv, YZ);
    Jac<Fq> r;
    r.x = fq_sub(Fv, fq_dbl(D));
    const Fq dx = fq_sub(D, r.x);
    pair_mul(E, dx, E, dx, M, unused);
    r.y = fq_sub(M, fq_dbl(fq_dbl(fq_dbl(C))));
    r.z = fq_dbl(YZ);
    return r;
}
__device__ __noinline__ Jac<Fq> jac_add_affine_pair(const Jac<Fq>& p, const G1A& q) {  // same formulas and cases as jac_add_affine
    if (affine_is_identity(q)) return p;
    if (fq_is_zero(p.z)) return Jac<Fq>{q.x, q.y, fq_one()};
    Fq zz, yz, u2, s2, hh, zh, hhh, v, r2, yh, M, unused;
    pair_mul(p.z, p.z, q.y, p.z, zz, yz);
    pair_mul(q.x, zz, yz, zz, u2, s2);
    const Fq h = fq_sub(u2, p.x), rr = fq_sub(s2, p.y);
    if (fq_is_zero(h)) {
        if (fq_is_zero(rr)) return jac_dbl_pair(p);
        return jac_identity<Fq>();
    }
    pair_mul(h, h, p.z, h, hh, zh);
    pair_mul(hh, h, p.x, hh, hhh, v);
    pair_mul(rr, rr, p.y, hhh, r2, yh);
    Jac<Fq> r;
    r.x = fq_sub(fq_sub(fq_sub(r2, hhh), v), v);
    const Fq vx = fq_sub(v, r.x);
    pair_mul(rr, vx, rr, vx, M, unused);
    r.y = fq_sub(M, yh);
    r.z = zh;
    return r;
}
__device__ __forceinline__ Jac<Fq> jac_scalar_mul_naf_pair(const G1A& q, const uint32_t* plus, const uint32_t* minus, int bits) {
    Jac<Fq> acc = jac_identity<Fq>();
    for (int i = bits - 1; i >= 0; i--) {
        acc = jac_dbl_pair(acc);
        const uint32_t m = 1u << (i & 31);
        const bool dp = (plus[i >> 5] & m) != 0, dm = (minus[i >> 5] & m) != 0;
        if (dp || dm) {
            G1A t = q;
            if (dm) t.y = fq_neg(q.y);
            acc = jac_add_affine_pair(acc, t);
        }
    }
    return acc;
}

// [k_j] (+-) endo^j(p2) for this warp's component
template <class F>
__device__ __forceinline__ Jac<F> fold_component(const Affine<F>& p2, const FoldComp& c, int j, int bits) {
    Affine<F> q = endo_apply(p2, j);
    if (c.neg) q.y = f_neg(q.y);
    return jac_scalar_mul_naf(q, c.plus, c.minus, bits);
}

__global__ void __launch_bounds__(SIPP_FOLD_THREADS) k_fold_split(uint32_t* __restrict__ A, uint32_t* __restrict__ B, size_t h, FoldPlan plan_arg,
                                                                 unsigned g2_blocks) {
    __shared__ FoldPlan plan;
    __shared__ __align__(16) uint32_t xch[3 * 32 * 48];  // G2: [3 comps][32 lanes][48 words]; G1: [2 halves][32 lanes][24 words]
    for (int i = threadIdx.x; i < (int)(sizeof(FoldPlan) / 4); i += blockDim.x) ((uint32_t*)&plan)[i] = ((const uint32_t*)&plan_arg)[i];
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (blockIdx.x < g2_blocks) {
        // 16 elements per block, every Fq2 on a PAIR of lanes (fq2h.cuh): an Fq2 product is one lazy inner product per lane
        // instead of three dependent Fq products on one thread -- the 66-doubling chain of a component gets ~1.75x shorter
        const int el = lane >> 1;
        size_t i = (size_t)blockIdx.x * 16 + el;
        const bool valid = i < h;
        if (!valid) i = h - 1;
        G2A q = endo_apply(load_g2(B, i + h), warp);
        if (plan.g2[warp].neg) q.y = f_neg(q.y);
        Jac<Fq2H> acc = jac_scalar_mul_naf(split_g2(q), plan.g2[warp].plus, plan.g2[warp].minus, plan.g2_bits);
        if (warp > 0) store_jac_h(xch + ((warp - 1) * 16 + el) * 48, acc);
        __syncthreads();
        if (warp == 0) {
#pragma unroll 1
            for (int j = 0; j < 3; j++) acc = jac_add(acc, load_jac_h(xch + (j * 16 + el) * 48));
            const Affine<Fq2H> r = jac_to_affine(jac_add_affine(acc, split_g2(load_g2(B, i))));
            if (valid) {
                const int o = h_odd() ? 8 : 0;
                store_fq_words(B + 32 * i + o, r.x.v);
                store_fq_words(B + 32 * i + 16 + o, r.y.v);
            }
        }
    } else {
        // 32 elements per block: warps (0, 1) and (2, 3) hold the two GLV components of 16 elements each, every element on a lane pair
        const int comp = warp & 1, half = warp >> 1, el = lane >> 1;
        size_t i = (size_t)(blockIdx.x - g2_blocks) * 32 + half * 16 + el;
        const bool valid = i < h;
        if (!valid) i = h - 1;
        G1A q = endo_apply(load_g1(A, i + h), comp);
        if (plan.g1[comp].neg) q.y = fq_neg(q.y);
        Jac<Fq> acc = jac_scalar_mul_naf_pair(q, plan.g1[comp].plus, plan.g1[comp].minus, plan.g1_bits);
        if (comp == 1 && !h_odd()) store_jac(xch + (half * 16 + el) * 24, acc);
        __syncthreads();
        if (comp == 0 && !h_odd()) {
            acc = jac_add(acc, load_jac1(xch + (half * 16 + el) * 24));
            G1A r = jac_to_affine(jac_add_affine(acc, load_g1(A, i)));
            if (valid) store_g1(A, i, r);
        }
    }
}


// Batched instances: the same lane split, but every instance has its own challenge, so the plan is read per element
// (plans[inst]).  A warp's 32 elements belong to one instance while h >= 32 (uniform digit tests); in the last rounds a warp
// spans several instances and the digit branches diverge -- those rounds hold 31/127 of an instance's fold work.
// The element mapping is a template parameter (fold_map.cuh): UniformFold for the lock-step batch, RaggedFold for the ragged one.
template <class Map>
__device__ __forceinline__ void fold_batch_body(uint32_t* __restrict__ A, uint32_t* __restrict__ B, const Map& map, const FoldPlan* __restrict__ plans,
                                                unsigned g2_blocks) {
    __shared__ __align__(16) uint32_t xch[3 * 16 * 48];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, el = lane >> 1;
    const size_t total = map.total();
    if (blockIdx.x < g2_blocks) {
        // as k_fold_split: 16 elements per block, every Fq2 on a lane pair; pairs of one warp may follow different digit schedules
        // (different instances) -- the pair shuffles of fq2h.cuh name only their own two lanes
        size_t e = (size_t)blockIdx.x * 16 + el;
        const bool valid = e < total;
        if (!valid) e = total - 1;
        const FoldElem fe = map.elem(e);
        const size_t i = fe.i, h = fe.h;
        const FoldPlan* pl = plans + fe.inst;
        G2A q = endo_apply(load_g2(B, i + h), warp);
        if (pl->g2[warp].neg) q.y = f_neg(q.y);
        Jac<Fq2H> acc = jac_scalar_mul_naf(split_g2(q), pl->g2[warp].plus, pl->g2[warp].minus, pl->g2_bits);
        if (warp > 0) store_jac_h(xch + ((warp - 1) * 16 + el) * 48, acc);
        __syncthreads();
        if (warp == 0) {
#pragma unroll 1
            for (int j = 0; j < 3; j++) acc = jac_add(acc, load_jac_h(xch + (j * 16 + el) * 48));
            const Affine<Fq2H> r = jac_to_affine(jac_add_affine(acc, split_g2(load_g2(B, i))));
            if (valid) {
                const int o = h_odd() ? 8 : 0;
                store_fq_words(B + 32 * i + o, r.x.v);
                store_fq_words(B + 32 * i + 16 + o, r.y.v);
            }
        }
    } else {
        const int comp = warp & 1, half = warp >> 1;
        size_t e = (size_t)(blockIdx.x - g2_blocks) * 32 + half * 16 + el;
        const bool valid = e < total;
        if (!valid) e = total - 1;
        const FoldElem fe = map.elem(e);
        const size_t i = fe.i, h = fe.h;
        const FoldPlan* pl = plans + fe.inst;
        G1A q = endo_apply(load_g1(A, i + h), comp);
        if (pl->g1[comp].neg) q.y = fq_neg(q.y);
        Jac<Fq> acc = jac_scalar_mul_naf_pair(q, pl->g1[comp].plus, pl->g1[comp].minus, pl->g1_bits);
        if (comp == 1 && !h_odd()) store_jac(xch + (half * 16 + el) * 24, acc);
        __syncthreads();
        if (comp == 0 && !h_odd()) {
            acc = jac_add(acc, load_jac1(xch + (half * 16 + el) * 24));
            G1A r = jac_to_affine(jac_add_affine(acc, load_g1(A, i)));
            if (valid) store_g1(A, i, r);
        }
    }
}
__global__ void __launch_bounds__(SIPP_FOLD_THREADS) k_fold_batch(uint32_t* __restrict__ A, uint32_t* __restrict__ B, size_t h, size_t stride, size_t count,
                                                                 const FoldPlan* __restrict__ plans, unsigned g2_blocks) {
    fold_batch_body(A, B, UniformFold{h, stride, count}, plans, g2_blocks);
}
__global__ void __launch_bounds__(SIPP_FOLD_THREADS) k_fold_batch_ragged(uint32_t* __restrict__ A, uint32_t* __restrict__ B, const RaggedInst* __restrict__ tab,
                                                                        unsigned act, size_t elems, const FoldPlan* __restrict__ plans, unsigned g2_blocks) {
    fold_batch_body(A, B, RaggedFold{tab, act, elems, 0}, plans, g2_blocks);
}

// ------------------------------------------------------------------------------------------------ K4, throughput form
// One thread per element, all endomorphism components on ONE accumulator (Straus / Shamir): the 66 (G2) or 128 (G1)
// doublings are shared by the 4 (2) sub-scalars instead of being repeated per component as in the lane-split kernels --
// G2: 66 dbl + ~88 mixed adds (~3.7k Fq-mul) against 4 x (66 dbl + 22 adds) (~6.9k); G1: ~1.8k against ~2.7k.  The lane
// split buys latency (k_fold_split / k_fold_wide, small rounds of one proof); this one buys work, for launches that fill
// the GPU: batched instances and the first rounds of a large proof.  plans[inst] as in k_fold_batch (count = 1: one proof).
#define SIPP_STRAUS_THREADS 64

template <class Map>
__device__ __forceinline__ void fold_straus_body(uint32_t* __restrict__ A, uint32_t* __restrict__ B, const Map& map, const FoldPlan* __restrict__ plans,
                                                 unsigned g2_blocks) {
    const size_t total = map.total();
    const bool is_g2 = blockIdx.x < g2_blocks;
    size_t e = (size_t)(is_g2 ? blockIdx.x : blockIdx.x - g2_blocks) * SIPP_STRAUS_THREADS + threadIdx.x;
    if (e >= total) return;
    const FoldElem fe = map.elem(e);
    const size_t i = fe.i, h = fe.h;
    const FoldPlan* pl = plans + fe.inst;
    if (is_g2) {
        G2A tbl[4];
        const G2A p2 = load_g2(B, i + h);
#pragma unroll 1
        for (int c = 0; c < 4; c++) {
            tbl[c] = endo_apply(p2, c);
            if (pl->g2[c].neg) tbl[c].y = f_neg(tbl[c].y);
        }
        Jac<Fq2> acc = straus_naf<Fq2, 4>(tbl, pl->g2, pl->g2_bits);
        store_g2(B, i, jac_to_affine(jac_add_affine(acc, load_g2(B, i))));
    } else {
        G1A tbl[2];
        const G1A p2 = load_g1(A, i + h);
#pragma unroll 1
        for (int c = 0; c < 2; c++) {
            tbl[c] = endo_apply(p2, c);
            if (pl->g1[c].neg) tbl[c].y = f_neg(tbl[c].y);
        }
        Jac<Fq> acc = straus_naf<Fq, 2>(tbl, pl->g1, pl->g1_bits);
        store_g1(A, i, jac_to_affine(jac_add_affine(acc, load_g1(A, i))));
    }
}
__global__ void __launch_bounds__(SIPP_STRAUS_THREADS) k_fold_straus(uint32_t* __restrict__ A, uint32_t* __restrict__ B, size_t h, size_t stride, size_t count,
                                                                   const FoldPlan* __restrict__ plans, unsigned g2_blocks) {
    fold_straus_body(A, B, UniformFold{h, stride, count}, plans, g2_blocks);
}
__global__ void __launch_bounds__(SIPP_STRAUS_THREADS) k_fold_straus_ragged(uint32_t* __restrict__ A, uint32_t* __restrict__ B, const RaggedInst* __restrict__ tab,
                                                                          unsigned act, size_t elems, const FoldPlan* __restrict__ plans, unsigned g2_blocks) {
    fold_straus_body(A, B, RaggedFold{tab, act, elems, 0}, plans, g2_blocks);
}

// ------------------------------------------------------------------------------------------------ input validation
// What `G1Affine::new` / `G2Affine::new` assert when the reference's inputs are built (on the curve, in the prime-order
// subgroup) -- checked here because the folds rely on it: psi is used as [6x^2] and phi as [lambda], which holds only in the
// r-torsion.  Thread t < n checks A_t: y^2 = x^3 + 3 (G1 has cofactor 1).  Thread n + i checks B_i: y^2 = x^3 + 3/xi and
//   [x + 1] Q + psi([x] Q) + psi^2([x] Q) == psi^3([2x] Q)     (x the BN parameter: one 63-bit scalar multiplication)
// which holds exactly for the points of order r (El Housni, Guillevic, Piellard 2022; tests/test_gpu_parity.py checks it on
// points of the twist outside G2).  The identity (x = y = 0, ark's `infinity`) passes.  flags |= 2: off the curve, |= 4: on
// the twist but outside G2.  Inputs are Montgomery limbs (after k_codec_decode).
__device__ __forceinline__ Jac<Fq2> psi_jac(const Jac<Fq2>& p, int j) {  // psi^j on Jacobian coordinates (Z^p = conj(Z))
    Jac<Fq2> r;
    r.x = f_mul((j & 1) ? fq2_conj(p.x) : p.x, frob_gamma(j, 2));
    r.y = f_mul((j & 1) ? fq2_conj(p.y) : p.y, frob_gamma(j, 3));
    r.z = (j & 1) ? fq2_conj(p.z) : p.z;
    return r;
}
__device__ bool jac_equal(const Jac<Fq2>& p, const Jac<Fq2>& q) {
    const bool pz = f_is_zero(p.z), qz = f_is_zero(q.z);
    if (pz || qz) return pz && qz;
    const Fq2 z1 = f_sqr(p.z), z2 = f_sqr(q.z);
    if (!fq2_eq(f_mul(p.x, z2), f_mul(q.x, z1))) return false;
    return fq2_eq(f_mul(p.y, f_mul(z2, q.z)), f_mul(q.y, f_mul(z1, p.z)));
}
__global__ void __launch_bounds__(64) k_validate_points(const uint32_t* __restrict__ dA, size_t n, const uint32_t* __restrict__ dB, size_t nb,
                                                         int* __restrict__ flags) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n + nb) return;
    if (t < n) {
        const G1A p{load_fq_words(dA + 16 * t), load_fq_words(dA + 16 * t + 8)};
        if (affine_is_identity(p)) return;
        const Fq three = fq_to_mont(Fq{{3, 0, 0, 0, 0, 0, 0, 0}});
        if (!f_is_zero(f_sub(f_sqr(p.y), f_add(f_mul(f_sqr(p.x), p.x), three)))) atomicOr(flags, 2);
        return;
    }
    const size_t i = t - n;
    const G2A q{load_fq2_words(dB + 32 * i), load_fq2_words(dB + 32 * i + 16)};
    if (affine_is_identity(q)) return;
    if (!fq2_eq(f_sqr(q.y), f_add(f_mul(f_sqr(q.x), q.x), fq2_b_twist()))) { atomicOr(flags, 2); return; }
    const unsigned long long xb = SIPP_BN_X;
    const uint32_t k[8] = {(uint32_t)xb, (uint32_t)(xb >> 32), 0, 0, 0, 0, 0, 0};
    const Jac<Fq2> xq = jac_scalar_mul(q, k);
    Jac<Fq2> lhs = jac_add_affine(xq, q);
    lhs = jac_add(lhs, psi_jac(xq, 1));
    lhs = jac_add(lhs, psi_jac(xq, 2));
    const Jac<Fq2> rhs = psi_jac(jac_dbl(xq), 3);
    if (!jac_equal(lhs, rhs)) atomicOr(flags, 4);
}
int launch_validate_points(const uint32_t* dA, const uint32_t* dB, size_t n, int* flags, cudaStream_t s) {
    return launch_validate_points_groups(dA, n, dB, n, flags, s);
}
int launch_validate_points_groups(const uint32_t* dA, size_t na, const uint32_t* dB, size_t nb, int* flags, cudaStream_t s) {
    k_validate_points<<<(unsigned)((na + nb + 63) / 64), 64, 0, s>>>(dA, na, dB, nb, flags);
    return (int)cudaGetLastError();
}

int launch_fold(uint32_t* A, uint32_t* B, size_t h, const FoldPlan& plan, cudaStream_t s) {
    // In-place: an element's partner i + h is only read by the block that owns i, and i < h <= i + h, so no block reads
    // what another block writes.
    unsigned g2_blocks = (unsigned)((h + 15) / 16), g1_blocks = (unsigned)((h + 31) / 32);
    k_fold_split<<<g2_blocks + g1_blocks, SIPP_FOLD_THREADS, 0, s>>>(A, B, h, plan, g2_blocks);
    return (int)cudaGetLastError();
}
int launch_fold_batch(uint32_t* A, uint32_t* B, size_t h, size_t stride, size_t count, const FoldPlan* plans, cudaStream_t s) {
    size_t total = count * h;
    unsigned g2_blocks = (unsigned)((total + 15) / 16), g1_blocks = (unsigned)((total + 31) / 32);
    k_fold_batch<<<g2_blocks + g1_blocks, SIPP_FOLD_THREADS, 0, s>>>(A, B, h, stride, count, plans, g2_blocks);
    return (int)cudaGetLastError();
}
int launch_fold_batch_ragged(uint32_t* A, uint32_t* B, const RaggedInst* tab, unsigned act, size_t elems, const FoldPlan* plans, cudaStream_t s) {
    unsigned g2_blocks = (unsigned)((elems + 15) / 16), g1_blocks = (unsigned)((elems + 31) / 32);
    k_fold_batch_ragged<<<g2_blocks + g1_blocks, SIPP_FOLD_THREADS, 0, s>>>(A, B, tab, act, elems, plans, g2_blocks);
    return (int)cudaGetLastError();
}
int launch_fold_straus_ragged(uint32_t* A, uint32_t* B, const RaggedInst* tab, unsigned act, size_t elems, const FoldPlan* plans, cudaStream_t s) {
    unsigned blocks = (unsigned)((elems + SIPP_STRAUS_THREADS - 1) / SIPP_STRAUS_THREADS);
    k_fold_straus_ragged<<<2 * blocks, SIPP_STRAUS_THREADS, 0, s>>>(A, B, tab, act, elems, plans, blocks);
    return (int)cudaGetLastError();
}
int launch_fold_straus(uint32_t* A, uint32_t* B, size_t h, size_t stride, size_t count, const FoldPlan* plans, cudaStream_t s) {
    size_t total = count * h;
    unsigned blocks = (unsigned)((total + SIPP_STRAUS_THREADS - 1) / SIPP_STRAUS_THREADS);
    k_fold_straus<<<2 * blocks, SIPP_STRAUS_THREADS, 0, s>>>(A, B, h, stride, count, plans, blocks);
    return (int)cudaGetLastError();
}

}  // namespace sipp

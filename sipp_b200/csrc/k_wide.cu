// k_wide.cu -- k_lines_wide: the G2 side of the Miller loop with 16 lanes per pair (engine.cuh), for the latency-bound
// rounds.  Same inputs and the same line table as k_lines (k_coop.cu): lines[prod][pair][91][80 words], so k_accum
// consumes either.  Lines differ from k_lines' by Fq2 factors only (projective scaling), which the final
// exponentiation removes; Z, Z_L, Z_R are bit-identical (tests/test_gpu_parity.py::test_wide_lines_*).
//
// Replaces the per-pair `pairing` calls of /root/reference/src/prover_native.rs:17-22, :48-49 (G2 arithmetic part).
#include "engine.cuh"
#include "device_common.cuh"
#include "fold_map.cuh"

namespace sipp {

#define SIPP_WIDE_THREADS 128
#define SIPP_WIDE_GROUPS (SIPP_WIDE_THREADS / SIPP_LP_LANES)
#define SIPP_LINE_WORDS 80

static __device__ const LpIns d_lp_code[SIPP_LP_LEVELS * SIPP_LP_LANES] = SIPP_LP_CODE_INIT;
static __constant__ unsigned char c_lp_types[SIPP_LP_LEVELS] = SIPP_LP_TYPES_INIT;

struct DevMachine {
    uint32_t* slots;
    uint32_t* out;  // line table of this pair
    int lane;
    bool store, ident;
    __device__ __forceinline__ void run(int first, int n) {
#pragma unroll 1
        for (int L = first; L < first + n; L++) {
            const uint4 w = __ldg(reinterpret_cast<const uint4*>(d_lp_code) + L * SIPP_LP_LANES + lane);
            const LpIns ins{w.x, w.y, w.z, w.w};
            const Fq r = lp_eval(c_lp_types[L], ins, slots);
            __syncwarp();  // every lane of the level has read its operands
            lp_store(slots, lp_dst(ins), r);
            __syncwarp();
        }
    }
    __device__ __forceinline__ void emit(int step) {
        if (lane < 10 && store) {
            Fq v = lp_load(slots, SIPP_LP_SLOT_OUT0 + lane);
            if (ident) v = (lane == 0) ? fq_one() : fq_zero();  // identity input: the pair contributes the factor 1
            uint4* o = reinterpret_cast<uint4*>(out + (size_t)step * SIPP_LINE_WORDS + lane * 8);
            o[0] = make_uint4(v.l[0], v.l[1], v.l[2], v.l[3]);
            o[1] = make_uint4(v.l[4], v.l[5], v.l[6], v.l[7]);
        }
    }
};

__global__ void __launch_bounds__(SIPP_WIDE_THREADS) k_lines_wide(const uint32_t* __restrict__ A, const uint32_t* __restrict__ B, MillerJob job, int nprod,
                                                                 size_t c0, size_t mc, uint32_t* __restrict__ lines) {
    __shared__ __align__(16) uint32_t smem[SIPP_WIDE_GROUPS * SIPP_LP_SLOTS * 8];
    __shared__ int ident_flag[SIPP_WIDE_GROUPS];
    const int group = threadIdx.x / SIPP_LP_LANES, lane = threadIdx.x % SIPP_LP_LANES;
    const size_t total = mc * (size_t)nprod;
    size_t t = (size_t)blockIdx.x * SIPP_WIDE_GROUPS + group;
    const bool valid = t < total;
    if (!valid) t = total - 1;  // surplus groups shadow the last pair (uniform control flow), nothing is stored
    const int prod = (int)(t / mc);
    const size_t j = c0 + (t - (size_t)prod * mc);
    uint32_t* slots = smem + group * (SIPP_LP_SLOTS * 8);
    if (lane == 0) {
        const G1A p = load_g1(A, job.a_off[prod] + j);
        const G2A q = load_g2(B, job.b_off[prod] + j);
        ident_flag[group] = (affine_is_identity(p) || affine_is_identity(q)) ? 1 : 0;
        lp_fill_fixed(slots, p.x, p.y, q.x, q.y);
    }
    __syncwarp();
    DevMachine mach;
    mach.slots = slots;
    mach.out = lines + t * (size_t)(SIPP_LINES_PER_PAIR * SIPP_LINE_WORDS);
    mach.lane = lane;
    mach.store = valid;
    mach.ident = ident_flag[group] != 0;
    lp_miller(mach);
}

// batched instances (launch.h BatchJob): same engine, pair index decomposed as (product, pair) like k_lines_batch -- the late rounds
// of a batch that does not fill the GPU with one thread per pair (a launch of a few thousand pairs takes the length of the
// per-thread chain, 1.8 ms, whatever its size; 16 lanes per pair bring it to 0.4 ms)
__global__ void __launch_bounds__(SIPP_WIDE_THREADS) k_lines_wide_batch(const uint32_t* __restrict__ A, const uint32_t* __restrict__ B, BatchJob job, size_t p0,
                                                                       size_t np, uint32_t* __restrict__ lines) {
    __shared__ __align__(16) uint32_t smem[SIPP_WIDE_GROUPS * SIPP_LP_SLOTS * 8];
    __shared__ int ident_flag[SIPP_WIDE_GROUPS];
    const int group = threadIdx.x / SIPP_LP_LANES, lane = threadIdx.x % SIPP_LP_LANES;
    const size_t total = np * job.h;
    size_t t = (size_t)blockIdx.x * SIPP_WIDE_GROUPS + group;
    const bool valid = t < total;
    if (!valid) t = total - 1;  // surplus groups shadow the last pair (uniform control flow), nothing is stored
    const size_t P = p0 + t / job.h, i = t % job.h;
    const size_t inst = P / (size_t)job.nprod;
    const int y = (int)(P % (size_t)job.nprod);
    const size_t base = inst * job.stride + i;
    uint32_t* slots = smem + group * (SIPP_LP_SLOTS * 8);
    if (lane == 0) {
        const G1A p = load_g1(A, base + job.a_off[y]);
        const G2A q = load_g2(B, base + job.b_off[y]);
        ident_flag[group] = (affine_is_identity(p) || affine_is_identity(q)) ? 1 : 0;
        lp_fill_fixed(slots, p.x, p.y, q.x, q.y);
    }
    __syncwarp();
    DevMachine mach;
    mach.slots = slots;
    mach.out = lines + t * (size_t)(SIPP_LINES_PER_PAIR * SIPP_LINE_WORDS);
    mach.lane = lane;
    mach.store = valid;
    mach.ident = ident_flag[group] != 0;
    lp_miller(mach);
}

int launch_lines_wide_batch(const uint32_t* A, const uint32_t* B, const BatchJob& job, size_t p0, size_t np, uint32_t* lines, cudaStream_t s) {
    const size_t groups = np * job.h;
    k_lines_wide_batch<<<(unsigned)((groups + SIPP_WIDE_GROUPS - 1) / SIPP_WIDE_GROUPS), SIPP_WIDE_THREADS, 0, s>>>(A, B, job, p0, np, lines);
    return (int)cudaGetLastError();
}

int launch_lines_wide(const uint32_t* A, const uint32_t* B, const MillerJob& job, int nprod, size_t c0, size_t mc, uint32_t* lines, cudaStream_t s) {
    const size_t groups = mc * (size_t)nprod;
    k_lines_wide<<<(unsigned)((groups + SIPP_WIDE_GROUPS - 1) / SIPP_WIDE_GROUPS), SIPP_WIDE_THREADS, 0, s>>>(A, B, job, nprod, c0, mc, lines);
    return (int)cudaGetLastError();
}

}  // namespace sipp

// ------------------------------------------------------------------------------------------------ K4 on the line engine
// k_fold_wide: the fixed-scalar fold of the latency-bound rounds.  As in k_fold_split the challenge is recoded on the host
// (fold_plan.h: GLS components for G2, GLV for G1, NAF digits) and one component = one scalar multiplication; here every
// component of every element gets a GROUP of 16 lanes that runs the generated point programs (DBL / ADD_P / ADD_M, the same
// tables as the Miller-loop lines; DBL1 / ADD1_* over Fq for G1), so a doubling is 2 MUL levels instead of ~16 dependent Fq
// products.  The two groups of a warp work on the SAME component of two elements: the digit schedule is warp-uniform.
//   A_i <- A_i + x A_{i+h}       /root/reference/src/prover_native.rs:60-64
//   B_i <- B_i + x^-1 B_{i+h}    /root/reference/src/prover_native.rs:65-69
// The component sums, the addition of the base point (all exceptional cases: identity, doubling, inverse) and the affine
// normalisation are the complete Jacobian formulas of curve.cuh, one thread per element.
namespace sipp {

__device__ __forceinline__ void store_words(uint32_t* dst, const Fq& v) {
#pragma unroll
    for (int i = 0; i < 8; i++) dst[i] = v.l[i];
}
__device__ __forceinline__ Fq load_words(const uint32_t* src) {
    Fq v;
#pragma unroll
    for (int i = 0; i < 8; i++) v.l[i] = src[i];
    return v;
}

__global__ void __launch_bounds__(SIPP_WIDE_THREADS) k_fold_wide(uint32_t* __restrict__ A, uint32_t* __restrict__ B, size_t h, FoldPlan plan_arg, unsigned g2_blocks) {
    __shared__ __align__(16) uint32_t smem[SIPP_WIDE_GROUPS * SIPP_LP_SLOTS * 8];
    __shared__ FoldPlan plan;
    __shared__ __align__(16) uint32_t xch[SIPP_WIDE_GROUPS * 48];  // one Jacobian point per group (G2: 48 words, G1: 24)
    for (int i = threadIdx.x; i < (int)(sizeof(FoldPlan) / 4); i += blockDim.x) ((uint32_t*)&plan)[i] = ((const uint32_t*)&plan_arg)[i];
    __syncthreads();
    const int warp = threadIdx.x >> 5, group = threadIdx.x / SIPP_LP_LANES, lane = threadIdx.x % SIPP_LP_LANES, gi = group & 1;
    uint32_t* slots = smem + group * (SIPP_LP_SLOTS * 8);
    DevMachine mach;
    mach.slots = slots; mach.out = nullptr; mach.lane = lane; mach.store = false; mach.ident = false;
    if (blockIdx.x < g2_blocks) {
        const int comp = warp;                       // 4 warps = 4 GLS components, 2 elements per block
        size_t e = (size_t)blockIdx.x * 2 + gi;
        const bool valid = e < h;
        if (!valid) e = h - 1;
        const FoldDigits d = fold_digits(plan.g2[comp], plan.g2_bits);
        bool ident = false;
        if (lane == 0) {
            G2A q = load_g2(B, e + h);
            ident = affine_is_identity(q);
            q = endo_apply(q, comp);
            if ((plan.g2[comp].neg != 0) != d.flip) q.y = fq2_neg(q.y);
            lp_fill_fixed(slots, fq_zero(), fq_zero(), q.x, q.y);
        }
        __syncwarp();
        if (d.top >= 0) {
            mach.run(SIPP_LP_SETUP_FIRST, SIPP_LP_SETUP_LEVELS);
            lp_scalar_mul(mach, true, d.plus, d.minus, d.top);
        }
        if (lane == 0) {
            Jac<Fq2> r = jac_identity<Fq2>();
            if (!ident && d.top >= 0) {
                const Fq2 X{lp_load(slots, SIPP_LP_SLOT_X0), lp_load(slots, SIPP_LP_SLOT_X1)}, Y{lp_load(slots, SIPP_LP_SLOT_Y0), lp_load(slots, SIPP_LP_SLOT_Y1)};
                const Fq2 Z = fq2_mul_xi(Fq2{lp_load(slots, SIPP_LP_SLOT_ZH0), lp_load(slots, SIPP_LP_SLOT_ZH1)});
                r.x = fq2_mul(X, Z);                 // homogeneous (X : Y : Z)  ->  Jacobian (X Z, Y Z^2, Z)
                r.y = fq2_mul(Y, fq2_sqr(Z));
                r.z = Z;
            }
            uint32_t* o = xch + group * 48;
            store_words(o, r.x.c0); store_words(o + 8, r.x.c1); store_words(o + 16, r.y.c0); store_words(o + 24, r.y.c1);
            store_words(o + 32, r.z.c0); store_words(o + 40, r.z.c1);
        }
        __syncthreads();
        if (warp == 0 && lane == 0) {
            Jac<Fq2> acc;
            for (int j = 0; j < 4; j++) {
                const uint32_t* o = xch + ((j * 2 + gi) * 48);   // group of component j, element gi
                Jac<Fq2> t;
                t.x = Fq2{load_words(o), load_words(o + 8)}; t.y = Fq2{load_words(o + 16), load_words(o + 24)}; t.z = Fq2{load_words(o + 32), load_words(o + 40)};
                acc = j ? jac_add(acc, t) : t;
            }
            const G2A r = jac_to_affine(jac_add_affine(acc, load_g2(B, e)));
            if (valid) store_g2(B, e, r);
        }
    } else {
        const int comp = warp & 1, pair = warp >> 1;  // warps (0,1) and (2,3): the two GLV components of 2 x 2 elements
        size_t e = (size_t)(blockIdx.x - g2_blocks) * 4 + pair * 2 + gi;
        const bool valid = e < h;
        if (!valid) e = h - 1;
        const FoldDigits d = fold_digits(plan.g1[comp], plan.g1_bits);
        bool ident = false;
        if (lane == 0) {
            G1A q = load_g1(A, e + h);
            ident = affine_is_identity(q);
            q = endo_apply(q, comp);
            if ((plan.g1[comp].neg != 0) != d.flip) q.y = fq_neg(q.y);
            lp_store(slots, SIPP_LP_SLOT_ZERO, fq_zero());
            lp_store(slots, SIPP_LP_SLOT_QX0, q.x); lp_store(slots, SIPP_LP_SLOT_QY0, q.y);
            lp_store(slots, SIPP_LP_SLOT_X1, q.x); lp_store(slots, SIPP_LP_SLOT_Y1, q.y); lp_store(slots, SIPP_LP_SLOT_Z1, fq_one());
        }
        __syncwarp();
        if (d.top >= 0) lp_scalar_mul(mach, false, d.plus, d.minus, d.top);
        if (lane == 0) {
            Jac<Fq> r = jac_identity<Fq>();
            if (!ident && d.top >= 0) {
                const Fq X = lp_load(slots, SIPP_LP_SLOT_X1), Y = lp_load(slots, SIPP_LP_SLOT_Y1), Z = lp_load(slots, SIPP_LP_SLOT_Z1);
                r.x = fq_mul(X, Z);
                r.y = fq_mul(Y, fq_sqr(Z));
                r.z = Z;
            }
            uint32_t* o = xch + group * 48;
            store_words(o, r.x); store_words(o + 8, r.y); store_words(o + 16, r.z);
        }
        __syncthreads();
        if (comp == 0 && lane == 0) {
            Jac<Fq> acc, t;
            const uint32_t* o0 = xch + group * 48;              // component 0 of this element
            const uint32_t* o1 = xch + (group + 2) * 48;        // component 1: next warp, same group-in-warp
            acc.x = load_words(o0); acc.y = load_words(o0 + 8); acc.z = load_words(o0 + 16);
            t.x = load_words(o1); t.y = load_words(o1 + 8); t.z = load_words(o1 + 16);
            acc = jac_add(acc, t);
            const G1A r = jac_to_affine(jac_add_affine(acc, load_g1(A, e)));
            if (valid) store_g1(A, e, r);
        }
    }
}

// batched instances: the plan is read per instance (plans[inst]); otherwise as k_fold_wide.  The element mapping is a template
// parameter (fold_map.cuh): UniformFold for the lock-step batch, RaggedFold for the ragged one.
template <class Map>
__device__ __forceinline__ void fold_wide_batch_body(uint32_t* __restrict__ A, uint32_t* __restrict__ B, const Map& map, const FoldPlan* __restrict__ plans,
                                                     unsigned g2_blocks) {
    __shared__ __align__(16) uint32_t smem[SIPP_WIDE_GROUPS * SIPP_LP_SLOTS * 8];
    __shared__ __align__(16) uint32_t xch[SIPP_WIDE_GROUPS * 48];  // one Jacobian point per group (G2: 48 words, G1: 24)
    // the two groups of a warp must run the same digit schedule: a unit is two elements of the SAME instance (h even: element pairs
    // start at even indices), or one element taken twice when h is odd (the second group is a shadow that stores nothing)
    const int warp = threadIdx.x >> 5, group = threadIdx.x / SIPP_LP_LANES, lane = threadIdx.x % SIPP_LP_LANES, gi = group & 1;
    uint32_t* slots = smem + group * (SIPP_LP_SLOTS * 8);
    DevMachine mach;
    mach.slots = slots; mach.out = nullptr; mach.lane = lane; mach.store = false; mach.ident = false;
    if (blockIdx.x < g2_blocks) {
        const int comp = warp;                       // 4 warps = 4 GLS components, 2 elements per block
        bool valid;
        const FoldElem fe = map.unit((size_t)blockIdx.x, gi, valid);
        const size_t e = fe.i, h = fe.h;
        const FoldPlan& plan = plans[fe.inst];
        const FoldDigits d = fold_digits(plan.g2[comp], plan.g2_bits);
        bool ident = false;
        if (lane == 0) {
            G2A q = load_g2(B, e + h);
            ident = affine_is_identity(q);
            q = endo_apply(q, comp);
            if ((plan.g2[comp].neg != 0) != d.flip) q.y = fq2_neg(q.y);
            lp_fill_fixed(slots, fq_zero(), fq_zero(), q.x, q.y);
        }
        __syncwarp();
        if (d.top >= 0) {
            mach.run(SIPP_LP_SETUP_FIRST, SIPP_LP_SETUP_LEVELS);
            lp_scalar_mul(mach, true, d.plus, d.minus, d.top);
        }
        if (lane == 0) {
            Jac<Fq2> r = jac_identity<Fq2>();
            if (!ident && d.top >= 0) {
                const Fq2 X{lp_load(slots, SIPP_LP_SLOT_X0), lp_load(slots, SIPP_LP_SLOT_X1)}, Y{lp_load(slots, SIPP_LP_SLOT_Y0), lp_load(slots, SIPP_LP_SLOT_Y1)};
                const Fq2 Z = fq2_mul_xi(Fq2{lp_load(slots, SIPP_LP_SLOT_ZH0), lp_load(slots, SIPP_LP_SLOT_ZH1)});
                r.x = fq2_mul(X, Z);                 // homogeneous (X : Y : Z)  ->  Jacobian (X Z, Y Z^2, Z)
                r.y = fq2_mul(Y, fq2_sqr(Z));
                r.z = Z;
            }
            uint32_t* o = xch + group * 48;
            store_words(o, r.x.c0); store_words(o + 8, r.x.c1); store_words(o + 16, r.y.c0); store_words(o + 24, r.y.c1);
            store_words(o + 32, r.z.c0); store_words(o + 40, r.z.c1);
        }
        __syncthreads();
        if (warp == 0 && lane == 0) {
            Jac<Fq2> acc;
            for (int j = 0; j < 4; j++) {
                const uint32_t* o = xch + ((j * 2 + gi) * 48);   // group of component j, element gi
                Jac<Fq2> t;
                t.x = Fq2{load_words(o), load_words(o + 8)}; t.y = Fq2{load_words(o + 16), load_words(o + 24)}; t.z = Fq2{load_words(o + 32), load_words(o + 40)};
                acc = j ? jac_add(acc, t) : t;
            }
            const G2A r = jac_to_affine(jac_add_affine(acc, load_g2(B, e)));
            if (valid) store_g2(B, e, r);
        }
    } else {
        const int comp = warp & 1, pair = warp >> 1;  // warps (0,1) and (2,3): the two GLV components of 2 x 2 elements
        bool valid;
        const FoldElem fe = map.unit((size_t)(blockIdx.x - g2_blocks) * 2 + pair, gi, valid);
        const size_t e = fe.i, h = fe.h;
        const FoldPlan& plan = plans[fe.inst];
        const FoldDigits d = fold_digits(plan.g1[comp], plan.g1_bits);
        bool ident = false;
        if (lane == 0) {
            G1A q = load_g1(A, e + h);
            ident = affine_is_identity(q);
            q = endo_apply(q, comp);
            if ((plan.g1[comp].neg != 0) != d.flip) q.y = fq_neg(q.y);
            lp_store(slots, SIPP_LP_SLOT_ZERO, fq_zero());
            lp_store(slots, SIPP_LP_SLOT_QX0, q.x); lp_store(slots, SIPP_LP_SLOT_QY0, q.y);
            lp_store(slots, SIPP_LP_SLOT_X1, q.x); lp_store(slots, SIPP_LP_SLOT_Y1, q.y); lp_store(slots, SIPP_LP_SLOT_Z1, fq_one());
        }
        __syncwarp();
        if (d.top >= 0) lp_scalar_mul(mach, false, d.plus, d.minus, d.top);
        if (lane == 0) {
            Jac<Fq> r = jac_identity<Fq>();
            if (!ident && d.top >= 0) {
                const Fq X = lp_load(slots, SIPP_LP_SLOT_X1), Y = lp_load(slots, SIPP_LP_SLOT_Y1), Z = lp_load(slots, SIPP_LP_SLOT_Z1);
                r.x = fq_mul(X, Z);
                r.y = fq_mul(Y, fq_sqr(Z));
                r.z = Z;
            }
            uint32_t* o = xch + group * 48;
            store_words(o, r.x); store_words(o + 8, r.y); store_words(o + 16, r.z);
        }
        __syncthreads();
        if (comp == 0 && lane == 0) {
            Jac<Fq> acc, t;
            const uint32_t* o0 = xch + group * 48;              // component 0 of this element
            const uint32_t* o1 = xch + (group + 2) * 48;        // component 1: next warp, same group-in-warp
            acc.x = load_words(o0); acc.y = load_words(o0 + 8); acc.z = load_words(o0 + 16);
            t.x = load_words(o1); t.y = load_words(o1 + 8); t.z = load_words(o1 + 16);
            acc = jac_add(acc, t);
            const G1A r = jac_to_affine(jac_add_affine(acc, load_g1(A, e)));
            if (valid) store_g1(A, e, r);
        }
    }
}
__global__ void __launch_bounds__(SIPP_WIDE_THREADS) k_fold_wide_batch(uint32_t* __restrict__ A, uint32_t* __restrict__ B, size_t h, size_t stride, size_t count,
                                                                      const FoldPlan* __restrict__ plans, unsigned g2_blocks) {
    fold_wide_batch_body(A, B, UniformFold{h, stride, count}, plans, g2_blocks);
}
__global__ void __launch_bounds__(SIPP_WIDE_THREADS) k_fold_wide_batch_ragged(uint32_t* __restrict__ A, uint32_t* __restrict__ B, const RaggedInst* __restrict__ tab,
                                                                             unsigned act, size_t elems, size_t units, const FoldPlan* __restrict__ plans,
                                                                             unsigned g2_blocks) {
    fold_wide_batch_body(A, B, RaggedFold{tab, act, elems, units}, plans, g2_blocks);
}

int launch_fold_wide_batch_ragged(uint32_t* A, uint32_t* B, const RaggedInst* tab, unsigned act, size_t elems, size_t units, const FoldPlan* plans,
                                  cudaStream_t s) {
    const unsigned g2_blocks = (unsigned)units, g1_blocks = (unsigned)((units + 1) / 2);
    k_fold_wide_batch_ragged<<<g2_blocks + g1_blocks, SIPP_WIDE_THREADS, 0, s>>>(A, B, tab, act, elems, units, plans, g2_blocks);
    return (int)cudaGetLastError();
}
int launch_fold_wide_batch(uint32_t* A, uint32_t* B, size_t h, size_t stride, size_t count, const FoldPlan* plans, cudaStream_t s) {
    const size_t total = count * h, epw = (h & 1) ? 1 : 2;
    const unsigned g2_blocks = (unsigned)((total + epw - 1) / epw), g1_blocks = (unsigned)((total + 2 * epw - 1) / (2 * epw));
    k_fold_wide_batch<<<g2_blocks + g1_blocks, SIPP_WIDE_THREADS, 0, s>>>(A, B, h, stride, count, plans, g2_blocks);
    return (int)cudaGetLastError();
}
int launch_fold_wide(uint32_t* A, uint32_t* B, size_t h, const FoldPlan& plan, cudaStream_t s) {
    const unsigned g2_blocks = (unsigned)((h + 1) / 2), g1_blocks = (unsigned)((h + 3) / 4);
    k_fold_wide<<<g2_blocks + g1_blocks, SIPP_WIDE_THREADS, 0, s>>>(A, B, h, plan, g2_blocks);
    return (int)cudaGetLastError();
}

}  // namespace sipp

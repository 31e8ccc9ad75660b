// k_mat.cu -- pairing-matrix stages of a single proof (host side: sipp_b200.cu mat_*; stage kinds and sizes: DESIGN.md section 4).
//
// The rounds of /root/reference/src/prover_native.rs:45-75 are a strictly serial chain of small launches: fold the points
// (:60-69), run the Miller loops of Z_L, Z_R (:48-49), exponentiate, hash, next challenge -- 2.7 ms per round on a GPU that is
// almost empty.  The chain is cut by bilinearity: with E[i][j] = e(A_i, B_j) for ALL pairs of the n points left -- or, with blocks
// of m points as "virtual points", E[i][j] = prod_t e(A[i m + t], B[j m + t]) -- computed in one launch set (the GPU has room),
//     Z_L = prod_{i<h} E[i+h][i],   Z_R = prod_{i<h} E[i][i+h]                                            (h = n / 2)
// and the fold A'_i = A_i + x A_{i+h}, B'_j = B_j + x^-1 B_{j+h} carries over to the matrix,
//     E'[i][j] = e(A'_i, B'_j) = E[i][j] * E[i+h][j+h] * E[i+h][j]^x * E[i][j+h]^(x^-1),
// two GT exponentiations per entry, each split by the Frobenius (p = 6x^2 mod r, the eigenvalue psi has on G2) into four
// 66-bit sub-scalars that run on their own 32-lane Fq12 machine with cyclotomic squarings -- so a tail round is ONE short
// kernel and a tiny product instead of fold + lines + accumulation + final exponentiation.  Pairing values are field elements:
// every Z_L, Z_R is bit-identical to the point-fold route (tests/test_gpu_parity.py: `pipeline` fixture, oracle, golden).
#include "device_common.cuh"
#include "machine12.cuh"

namespace sipp {

// pair q = (i * nr + j) * m + t of the expanded launch is (A[i m + t], B[j m + t]): entry (i, j) of the matrix owns m consecutive pairs
__global__ void k_mat_gather(const uint32_t* __restrict__ A, const uint32_t* __restrict__ B, size_t nr, size_t m, uint32_t* __restrict__ Aexp,
                             uint32_t* __restrict__ Bexp) {
    const size_t th = (size_t)blockIdx.x * blockDim.x + threadIdx.x;  // one uint4 (4 words) per thread: 4 + 8 per pair
    const size_t q = th / 12;
    const int w = (int)(th % 12);
    if (q >= nr * nr * m) return;
    const size_t e = q / m, t = q % m, i = e / nr, j = e % nr;
    if (w < 4) reinterpret_cast<uint4*>(Aexp + 16 * q)[w] = __ldg(reinterpret_cast<const uint4*>(A + 16 * (i * m + t)) + w);
    else reinterpret_cast<uint4*>(Bexp + 32 * q)[w - 4] = __ldg(reinterpret_cast<const uint4*>(B + 32 * (j * m + t)) + (w - 4));
}
int launch_mat_gather(const uint32_t* A, const uint32_t* B, size_t nr, size_t m, uint32_t* Aexp, uint32_t* Bexp, cudaStream_t s) {
    const size_t threads = nr * nr * m * 12;
    k_mat_gather<<<(unsigned)((threads + 255) / 256), 256, 0, s>>>(A, B, nr, m, Aexp, Bexp);
    return (int)cudaGetLastError();
}

// one machine (warp) per entry: the final exponentiation of a Miller value, left in HBM register-shaped (96 words, slot 2k + c,
// Montgomery) for the folds below
#define SIPP_MAT_FE_MACHINES 4
#define SIPP_MAT_FE_SLOTS (SIPP_F12_GLOBAL_SLOTS + SIPP_F12_REG_SLOTS * SIPP_F12_FE_REGS)
__global__ void __launch_bounds__(SIPP_MAT_FE_MACHINES * 32) k_mat_fe(const uint32_t* __restrict__ miller, size_t count, uint32_t* __restrict__ E, int ark_norm) {
    __shared__ __align__(16) uint32_t smem[SIPP_MAT_FE_MACHINES * SIPP_MAT_FE_SLOTS * 8];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t* slots = smem + warp * (SIPP_MAT_FE_SLOTS * 8);
    size_t q = (size_t)blockIdx.x * SIPP_MAT_FE_MACHINES + warp;
    const bool have = q < count;
    if (!have) q = count - 1;  // surplus machines shadow the last entry, nothing is stored
    for (int j = lane; j < 37; j += 32) f12_fill_global(slots, j);
    for (int w = lane; w < 96; w += 32) slots[f12_reg_base(0) * 8 + w] = miller[q * 96 + w];
    __syncwarp();
    DevMachine12 mc;
    mc.slots = slots;
    mc.lane = lane;
    const int res = f12_final_exp(mc, ark_norm != 0);
    if (have)
        for (int w = lane; w < 96; w += 32) E[q * 96 + w] = slots[f12_reg_base(res) * 8 + w];
}
int launch_mat_fe(const uint32_t* miller, size_t count, uint32_t* E, int ark_norm, cudaStream_t s) {
    k_mat_fe<<<(unsigned)((count + SIPP_MAT_FE_MACHINES - 1) / SIPP_MAT_FE_MACHINES), SIPP_MAT_FE_MACHINES * 32, 0, s>>>(miller, count, E, ark_norm);
    return (int)cudaGetLastError();
}

// the factors of Z_L, Z_R in the layout the reduction kernels read: partials[i][y][96], y = 0: E[i+h][i]  (inner_product(A2, B1),
// prover_native.rs:48), y = 1: E[i][i+h]  (inner_product(A1, B2), :49); main_diagonal: partials[i][96] = E[i][i], the factors of
// Z = inner_product(A, B)  (:29) when the first matrix is built from the inputs themselves
__global__ void k_mat_diag(const uint32_t* __restrict__ E, size_t n, int main_diagonal, uint32_t* __restrict__ partials) {
    const size_t h = n / 2;
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t e = t / 24;  // 24 uint4 per entry
    const int w = (int)(t % 24);
    if (e >= (main_diagonal ? n : 2 * h)) return;
    const size_t i = e >> 1;
    const int y = (int)(e & 1);
    const size_t src = main_diagonal ? e * n + e : (y == 0 ? (i + h) * n + i : i * n + (i + h));
    reinterpret_cast<uint4*>(partials + e * 96)[w] = __ldg(reinterpret_cast<const uint4*>(E + src * 96) + w);
}
int launch_mat_diag(const uint32_t* E, size_t n, int main_diagonal, uint32_t* partials, cudaStream_t s) {
    const size_t threads = n * 24;
    k_mat_diag<<<(unsigned)((threads + 127) / 128), 128, 0, s>>>(E, n, main_diagonal, partials);
    return (int)cudaGetLastError();
}

// k_mat_fold: one block per entry (i, j), i != j (all entries with `diag`), of the folded matrix; 8 machines = 2 exponents x 4 Frobenius components.
//   machine w < 4:  (frob^w E[i+h][j])^(k_w of x)        machine 4 + w:  (frob^w E[i][j+h])^(k_w of x^-1)
// then machine 0 multiplies E[i][j] in, machine 4 E[i+h][j+h], and a tree product over the eight leaves the entry in machine 0.
// The diagonal is never read by a later round (Z_L, Z_R use |i - j| = h / 2 and folds keep i - j modulo h), so it is skipped, unless
// `diag`: the statement prover reads the 1 x 1 matrix after the last round, <final_A, final_B>, which needs every diagonal before it.
#define SIPP_MAT_MACHINES 8
#define SIPP_MAT_REGS 4  // 0 accumulator, 1 base, 2 its conjugate, 3 exchange
#define SIPP_MAT_SLOTS (SIPP_F12_GLOBAL_SLOTS + SIPP_F12_REG_SLOTS * SIPP_MAT_REGS)
__global__ void __launch_bounds__(SIPP_MAT_MACHINES * 32) k_mat_fold(const uint32_t* __restrict__ E, size_t n, uint32_t* __restrict__ Eout, GtPlan plan_arg, int diag) {
    __shared__ __align__(16) uint32_t smem[SIPP_MAT_MACHINES * SIPP_MAT_SLOTS * 8];
    __shared__ GtPlan plan;
    const size_t h = n / 2;
    const size_t i = blockIdx.x / h, j = blockIdx.x % h;
    if (i == j && !diag) return;
    for (int t = threadIdx.x; t < (int)(sizeof(GtPlan) / 4); t += blockDim.x) ((uint32_t*)&plan)[t] = ((const uint32_t*)&plan_arg)[t];
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t* slots = smem + warp * (SIPP_MAT_SLOTS * 8);
    for (int t = lane; t < 37; t += 32) f12_fill_global(slots, t);
    auto load_reg = [&](int reg, size_t entry) {
        const uint4* src = reinterpret_cast<const uint4*>(E + entry * 96);
        if (lane < 24) reinterpret_cast<uint4*>(slots + f12_reg_base(reg) * 8)[lane] = __ldg(src + lane);
        __syncwarp();
    };
    const int which = warp >> 2, comp = warp & 3;
    load_reg(1, which == 0 ? (i + h) * n + j : i * n + (j + h));
    DevMachine12 mc;
    mc.slots = slots;
    mc.lane = lane;
    if (!f12_gt_pow_comp(mc, comp, plan.c[warp], plan.bits)) {  // zero sub-scalar: the factor 1
        if (lane < 12) lp_store(slots, f12_reg_base(0) + lane, lane == 0 ? fq_one() : fq_zero());
        __syncwarp();
    }
    if (comp == 0) {
        load_reg(3, which == 0 ? i * n + j : (i + h) * n + (j + h));
        F12_OP3(mc, MUL12, 0, 0, 3);
    }
#pragma unroll 1
    for (int half = SIPP_MAT_MACHINES / 2; half >= 1; half >>= 1) {
        __syncthreads();
        if (warp < half) {
            const uint32_t* other = smem + (warp + half) * (SIPP_MAT_SLOTS * 8) + f12_reg_base(0) * 8;
            for (int w = lane; w < 96; w += 32) slots[f12_reg_base(3) * 8 + w] = other[w];
            __syncwarp();
            F12_OP3(mc, MUL12, 0, 0, 3);
        }
    }
    if (warp == 0) {
        uint32_t* o = Eout + (i * h + j) * 96;
        for (int w = lane; w < 96; w += 32) o[w] = slots[f12_reg_base(0) * 8 + w];
    }
}
int launch_mat_fold(const uint32_t* E, size_t n, uint32_t* Eout, const GtPlan& plan, bool diag, cudaStream_t s) {
    const size_t h = n / 2;
    k_mat_fold<<<(unsigned)(h * h), SIPP_MAT_MACHINES * 32, 0, s>>>(E, n, Eout, plan, diag ? 1 : 0);
    return (int)cudaGetLastError();
}

}  // namespace sipp

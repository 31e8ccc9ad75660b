// msmcheck.cpp -- TEST HARNESS ONLY.  Compiles the recoding and bucket code of the multi-scalar multiplications
// (sipp_b200/csrc/msm.cuh, the functions k_msm.cu runs) for the host with g++, so that tests/test_msm_cpu.py can check them
// against the oracle without a GPU.  The lattice tables are the product's (glv_consts.h).  Never linked into the product.
#include <cstring>
#include <vector>

#include "../../sipp_b200/csrc/codec.cuh"
#include "../../sipp_b200/csrc/glv_consts.h"
#include "../../sipp_b200/csrc/msm.cuh"

using namespace sipp;

static const glv::Tables TABLES = {&SIPP_GLV_G1_BASIS[0][0][0], &SIPP_GLV_G1_RECIP[0][0], SIPP_GLV_G1_RECIP_SIGN,
                                   &SIPP_GLS_G2_BASIS[0][0][0], &SIPP_GLS_G2_RECIP[0][0], SIPP_GLS_G2_RECIP_SIGN};

static const uint32_t* W(const uint8_t* p) { return reinterpret_cast<const uint32_t*>(p); }
static uint32_t* W(uint8_t* p) { return reinterpret_cast<uint32_t*>(p); }

template <class F>
static int recode(const uint8_t* k, int c, int* negs, uint8_t* mags, int* digits) {
    constexpr int NC = msm::Group<F>::NC;
    FoldSubScalar sub[NC];
    if (!msm::scalar_below_r(W(k))) return -2;
    if (msm::split<F>(W(k), TABLES, sub)) return -1;
    const int nw = msm::windows(msm::Group<F>::BITS, c);
    for (int j = 0; j < NC; j++) {
        negs[j] = sub[j].neg;
        memcpy(mags + 24 * j, sub[j].mag, 24);
        msm::signed_digits(sub[j].mag, msm::Group<F>::BITS, c, [&](int w, int d) { digits[j * nw + w] = d; });
    }
    return nw;
}

// the MSM of n points through the kernels' functions: c = 0 Straus (NAF, shared doublings), else Pippenger with c-bit windows whose
// buckets are reduced in parts of `part` buckets (as k_msm_windows splits them over threads and blocks)
template <class F>
static int msm_host(const uint8_t* points, const uint8_t* scalars, size_t n, int c, int part, uint8_t* out) {
    constexpr int NC = msm::Group<F>::NC, BITS = msm::Group<F>::BITS, PB = (int)sizeof(Affine<F>);  // 64 B G1, 128 B G2
    std::vector<Affine<F>> terms(n * NC);
    std::vector<FoldComp> naf(n * NC);
    const int nw = c ? msm::windows(BITS, c) : 0;
    const uint32_t nb = c ? 1u << (c - 1) : 0;
    std::vector<std::vector<uint32_t>> buckets((size_t)nw * nb);
    for (size_t i = 0; i < n; i++) {
        FoldSubScalar sub[NC];
        if (!msm::scalar_below_r(W(scalars + 32 * i)) || msm::split<F>(W(scalars + 32 * i), TABLES, sub)) return -1;
        Affine<F> p;
        const uint32_t* pw = W(points + (size_t)PB * i);
        if constexpr (NC == 2) p = g1_decode(pw);
        else p = g2_decode(pw);
        for (int j = 0; j < NC; j++) {
            const uint32_t t = (uint32_t)(i * NC + j);
            terms[t] = msm::term_point(p, j, sub[j].neg);
            glv::naf(sub[j].mag, naf[t].plus, naf[t].minus);
            if (c)
                msm::signed_digits(sub[j].mag, BITS, c, [&](int w, int d) {
                    if (d) buckets[(size_t)w * nb + (uint32_t)(d < 0 ? -d : d) - 1].push_back(t << 1 | (d < 0 ? 1u : 0u));
                });
        }
    }
    Jac<F> acc;
    if (!c) {
        acc = msm::straus_terms(terms.data(), naf.data(), n * NC, BITS + 1);
    } else {
        // the sorted (bucket, entry) list of k_msm_recode + the radix sort, summed in chunks of `part` % 7 + 1 entries as
        // k_msm_chunks / k_msm_buckets do (small chunks: most buckets cross chunks)
        std::vector<uint32_t> keys, vals;
        for (size_t b = 0; b < buckets.size(); b++)
            for (uint32_t v : buckets[b]) { keys.push_back((uint32_t)b); vals.push_back(v); }
        const uint32_t nbk = (uint32_t)buckets.size(), ent = (uint32_t)keys.size(), ch = (uint32_t)(part % 7 + 1);
        for (int z = 0; z < 5; z++) { keys.push_back(nbk); vals.push_back(0); }  // zero digits sort last
        std::vector<Jac<F>> sums((size_t)nw * nb, jac_identity<F>()), wins(nw), first(ent + 5), last(ent + 5);
        for (uint32_t k = 0; k * ch < ent + 5; k++) msm::chunk_sums(keys.data(), vals.data(), ent + 5, nbk, k, ch, terms.data(), sums.data(), first.data(), last.data());
        // a bucket over more than 2 chunks goes the long way: its partials summed in another order (k_msm_long_buckets: strided, then a tree)
        for (uint32_t b = 0; b < nbk; b++) {
            if (msm::bucket_combine(keys.data(), ent + 5, b, ch, 2, first.data(), last.data(), sums.data())) continue;
            const uint32_t lo = msm::lower_bound(keys.data(), ent + 5, b), hi = msm::lower_bound(keys.data(), ent + 5, b + 1);
            const uint32_t kl = lo / ch, kh = (hi - 1) / ch;
            Jac<F> even = last[kl], odd = jac_identity<F>();
            for (uint32_t k = kl + 1; k <= kh; k++) (k & 1 ? odd : even) = jac_add(k & 1 ? odd : even, first[k]);
            sums[b] = jac_add(odd, even);
        }
        for (int w = 0; w < nw; w++) {
            wins[w] = jac_identity<F>();
            for (uint32_t lo = 0; lo < nb; lo += (uint32_t)part)
                wins[w] = jac_add(wins[w], msm::window_part(sums.data() + (size_t)w * nb, lo, lo + (uint32_t)part < nb ? lo + (uint32_t)part : nb));
        }
        acc = msm::combine_windows(wins.data(), nw, c);
    }
    const Affine<F> r = jac_to_affine(acc);
    if constexpr (NC == 2) g1_encode(W(out), r);
    else g2_encode(W(out), r);
    return 0;
}

extern "C" {
// group 1 / 2: sub-scalar signs (NC ints), magnitudes (NC x 24 B little-endian) and signed digits (NC x W ints); returns W, -1 when
// a sub-scalar does not fit its bound, -2 for k >= r
int hc_msm_recode(int group, const uint8_t* k, int c, int* negs, uint8_t* mags, int* digits) {
    return group == 1 ? recode<Fq>(k, c, negs, mags, digits) : recode<Fq2>(k, c, negs, mags, digits);
}
int hc_msm(int group, const uint8_t* points, const uint8_t* scalars, size_t n, int c, int part, uint8_t* out) {
    return group == 1 ? msm_host<Fq>(points, scalars, n, c, part, out) : msm_host<Fq2>(points, scalars, n, c, part, out);
}
}

// msm.cuh -- recoding and bucket arithmetic of the multi-scalar multiplications (k_msm.cu; C ABI in msm.cu), shared with the host
// harness tests/msmcheck so that both can be checked against the oracle without a GPU.
//
//   sum_i [k_i] P_i  with  k_i = sum_j (-1)^neg_j m_j L^j (mod r)   (glv_core.h: G1 2 x m_j < 2^128, G2 4 x m_j < 2^66)
//   = sum_i sum_j [m_j] T_ij,  T_ij = (-1)^neg_j endo^j(P_i)          (curve.cuh endo_apply: phi on G1, psi on G2)
// so an n-point 254-bit MSM is an NC n-term MSM with short scalars.  Each term is then written one of two ways:
//   Pippenger  signed c-bit digits d_w in [-(2^(c-1) - 1), 2^(c-1)], W = bits / c + 1 windows: bucket |d_w| - 1 of window w
//              collects +-T_ij; a window is sum_b (b + 1) S_b, the windows are combined with c doublings each
//   Straus     the non-adjacent form of m_j (glv::naf): one accumulator per segment, one doubling per digit shared by all its terms
#pragma once
#include "curve.cuh"
#include "glv_core.h"

namespace sipp {
namespace msm {

template <class F>
struct Group;
template <>
struct Group<Fq> {
    static constexpr int NC = 2;      // GLV components
    static constexpr int BITS = 128;  // every sub-scalar is < 2^BITS
};
template <>
struct Group<Fq2> {
    static constexpr int NC = 4;
    static constexpr int BITS = 66;
};

SIPP_HD int windows(int bits, int c) { return bits / c + 1; }

// k (8 little-endian u32 words) < r ?
SIPP_HD bool scalar_below_r(const uint32_t k[8]) {
    const uint32_t RL[8] = {0xf0000001u, 0x43e1f593u, 0x79b97091u, 0x2833e848u, 0x8181585du, 0xb85045b6u, 0xe131a029u, 0x30644e72u};
    for (int i = 7; i >= 0; i--)
        if (k[i] != RL[i]) return k[i] < RL[i];
    return false;
}

// k < r -> NC sub-scalars, each < 2^BITS; returns 0, or -1 when a sub-scalar does not fit (cannot happen for k < r)
template <class F>
SIPP_HD int split(const uint32_t k[8], const glv::Tables& t, FoldSubScalar out[Group<F>::NC]);
template <>
SIPP_HD int split<Fq>(const uint32_t k[8], const glv::Tables& t, FoldSubScalar out[2]) {
    uint64_t k64[4];
    for (int i = 0; i < 4; i++) k64[i] = (uint64_t)k[2 * i] | ((uint64_t)k[2 * i + 1] << 32);
    if (glv::decompose<2>(k64, t.g1_basis, t.g1_recip, t.g1_sign, out)) return -1;
    for (int j = 0; j < 2; j++)
        if (out[j].mag[2]) return -1;  // >= 2^128
    return 0;
}
template <>
SIPP_HD int split<Fq2>(const uint32_t k[8], const glv::Tables& t, FoldSubScalar out[4]) {
    uint64_t k64[4];
    for (int i = 0; i < 4; i++) k64[i] = (uint64_t)k[2 * i] | ((uint64_t)k[2 * i + 1] << 32);
    if (glv::decompose<4>(k64, t.g2_basis, t.g2_recip, t.g2_sign, out)) return -1;
    for (int j = 0; j < 4; j++)
        if (out[j].mag[2] || (out[j].mag[1] >> 2)) return -1;  // >= 2^66
    return 0;
}

// bits [pos, pos + c) of a 192-bit magnitude (c <= 32)
SIPP_HD uint32_t bits_at(const uint64_t mag[3], int pos, int c) {
    const int w = pos >> 6, s = pos & 63;
    if (w >= 3) return 0;
    uint64_t v = mag[w] >> s;
    if (s && w + 1 < 3) v |= mag[w + 1] << (64 - s);
    return (uint32_t)(v & ((1ull << c) - 1));
}

// the signed c-bit digits of a magnitude < 2^bits, least significant first: sum_w d[w] 2^(c w) = mag, |d[w]| <= 2^(c-1).
// `emit(w, d)` is called for every window w < windows(bits, c), zero digits included.
template <class Emit>
SIPP_HD void signed_digits(const uint64_t mag[3], int bits, int c, Emit emit) {
    const int W = windows(bits, c);
    const int half = 1 << (c - 1);
    int carry = 0;
    for (int w = 0; w < W; w++) {
        int d = (int)bits_at(mag, c * w, c) + carry;
        carry = d > half;
        if (carry) d -= 1 << c;
        emit(w, d);
    }
}

// GT (k_gt_msm.cu): unsigned c-bit digits of a scalar < r < 2^254, no split -- ceil(254 / c) windows of 2^c - 1 buckets (digit d > 0 in
// bucket d - 1).  Fq12 has no cheap inverse, and the multi-exponentiation is defined for every Fq12, not only for GT.
SIPP_HD int gt_windows(int c) { return (254 + c - 1) / c; }
// bits [pos, pos + c) of a 256-bit little-endian scalar (c <= 16)
SIPP_HD uint32_t scalar_digit(const uint32_t k[8], int pos, int c) {
    const int w = pos >> 5, s = pos & 31;
    uint64_t v = k[w] >> s;
    if (w + 1 < 8) v |= (uint64_t)k[w + 1] << (32 - s);
    return (uint32_t)(v & ((1ull << c) - 1));
}

// the term table entry of sub-scalar j: (-1)^neg endo^j(P)
template <class F>
SIPP_HD Affine<F> term_point(const Affine<F>& p, int j, int neg) {
    Affine<F> q = endo_apply(p, j);
    if (neg) q.y = f_neg(q.y);
    return q;
}

// a bucket entry: term index << 1 | sign of the digit
template <class F>
SIPP_HD Jac<F> bucket_sum(const Affine<F>* terms, const uint32_t* vals, size_t count) {
    Jac<F> acc = jac_identity<F>();
    for (size_t e = 0; e < count; e++) {
        Affine<F> q = terms[vals[e] >> 1];
        if (vals[e] & 1) q.y = f_neg(q.y);
        acc = jac_add_affine(acc, q);
    }
    return acc;
}

// first index e in [0, n) with keys[e] >= key
SIPP_HD uint32_t lower_bound(const uint32_t* keys, uint32_t n, uint32_t key) {
    uint32_t lo = 0, hi = n;
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (keys[mid] < key) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

// the segment of item i: the last segment whose first item is <= i (empty segments share their first with the next one)
template <class Seg>
SIPP_HD uint32_t segment_of(const Seg* segs, uint32_t count, uint32_t i) {
    uint32_t lo = 0, hi = count;  // invariant: segs[lo].first <= i, answer in [lo, hi)
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (segs[mid].first <= i) lo = mid;
        else hi = mid;
    }
    return lo;
}

// [v] P for a small non-negative integer v (Jacobian P), MSB first
template <class F>
SIPP_HD Jac<F> jac_mul_small(const Jac<F>& p, uint32_t v) {
    Jac<F> acc = jac_identity<F>();
    for (int i = 31; i >= 0; i--) {
        if (!f_is_zero(acc.z)) acc = jac_dbl(acc);
        if ((v >> i) & 1u) acc = jac_add(acc, p);
    }
    return acc;
}

// The bucket runs and window sums below are written once over a group in an Ops type: T (a bucket or partial), In (a table entry),
// identity(), add(a, b), run(terms, vals, count) (the sum of a run of >= 1 sorted entries) and mul_small(p, v) ([v] p).  JacOps is G1 /
// G2 in Jacobian coordinates; the GT multi-exponentiation (k_gt_msm.cu) writes the same logic multiplicatively over Fq12.
template <class F>
struct JacOps {
    using T = Jac<F>;
    using In = Affine<F>;
    static SIPP_HD T identity() { return jac_identity<F>(); }
    static SIPP_HD T add(const T& a, const T& b) { return jac_add(a, b); }
    static SIPP_HD T run(const In* terms, const uint32_t* vals, size_t count) { return bucket_sum(terms, vals, count); }
    static SIPP_HD T mul_small(const T& p, uint32_t v) { return jac_mul_small(p, v); }
};

// Bucket sums from the sorted entries in chunks of `ch` entries, so that no thread walks a whole bucket (the buckets of a window
// are far from even: the top window of a short sub-scalar uses few of them).  Chunk k sums every run of equal keys inside
// [k ch, (k + 1) ch): a run that is a whole bucket goes to buckets[key]; otherwise its first run goes to first[k] and its last run to
// last[k] (one run spanning the chunk is both).  Keys >= nbuckets (zero digits) are skipped.
template <class Ops>
SIPP_HD void chunk_sums_of(const uint32_t* keys, const uint32_t* vals, uint32_t entries, uint32_t nbuckets, uint32_t k, uint32_t ch,
                           const typename Ops::In* terms, typename Ops::T* buckets, typename Ops::T* first, typename Ops::T* last) {
    const uint32_t s = k * ch, e = s + ch < entries ? s + ch : entries;
    uint32_t r = s;
    while (r < e) {
        const uint32_t key = keys[r];
        uint32_t q = r;
        while (q < e && keys[q] == key) q++;
        if (key >= nbuckets) break;  // the zero-digit entries sort last
        const typename Ops::T acc = Ops::run(terms, vals + r, q - r);
        const bool whole = (r == 0 || keys[r - 1] != key) && (q == entries || keys[q] != key);
        if (whole) {
            buckets[key] = acc;
        } else {
            if (r == s) first[k] = acc;
            if (q == e) last[k] = acc;
        }
        r = q;
    }
}
template <class F>
SIPP_HD void chunk_sums(const uint32_t* keys, const uint32_t* vals, uint32_t entries, uint32_t nbuckets, uint32_t k, uint32_t ch,
                        const Affine<F>* terms, Jac<F>* buckets, Jac<F>* first, Jac<F>* last) {
    chunk_sums_of<JacOps<F>>(keys, vals, entries, nbuckets, k, ch, terms, buckets, first, last);
}

// bucket b when its run [lo, hi) crosses chunks: the last run of its first chunk, the whole chunks between, the first run of its last
// chunk (buckets inside one chunk were written by chunk_sums, empty ones stay the identity).  Returns false, writing nothing, when the
// run crosses more than max_span chunks: the caller sums those partials in parallel (k_msm_long_buckets), in any order.
template <class Ops>
SIPP_HD bool bucket_combine_of(const uint32_t* keys, uint32_t entries, uint32_t b, uint32_t ch, uint32_t max_span, const typename Ops::T* first,
                               const typename Ops::T* last, typename Ops::T* buckets) {
    const uint32_t lo = lower_bound(keys, entries, b), hi = lower_bound(keys, entries, b + 1);
    if (hi == lo || lo / ch == (hi - 1) / ch) return true;
    const uint32_t kl = lo / ch, kh = (hi - 1) / ch;
    if (kh - kl > max_span) return false;
    typename Ops::T acc = last[kl];
    for (uint32_t k = kl + 1; k <= kh; k++) acc = Ops::add(acc, first[k]);
    buckets[b] = acc;
    return true;
}
template <class F>
SIPP_HD bool bucket_combine(const uint32_t* keys, uint32_t entries, uint32_t b, uint32_t ch, uint32_t max_span, const Jac<F>* first,
                            const Jac<F>* last, Jac<F>* buckets) {
    return bucket_combine_of<JacOps<F>>(keys, entries, b, ch, max_span, first, last, buckets);
}

// sum_{lo <= b < hi} (b + 1) S_b of one window's buckets (running sums from the top, then lo times the plain sum)
template <class Ops>
SIPP_HD typename Ops::T window_part_of(const typename Ops::T* buckets, uint32_t lo, uint32_t hi) {
    typename Ops::T run = Ops::identity(), acc = Ops::identity();
    for (uint32_t b = hi; b > lo; b--) {
        run = Ops::add(run, buckets[b - 1]);
        acc = Ops::add(acc, run);
    }
    return lo ? Ops::add(acc, Ops::mul_small(run, lo)) : acc;
}
template <class F>
SIPP_HD Jac<F> window_part(const Jac<F>* buckets, uint32_t lo, uint32_t hi) {
    return window_part_of<JacOps<F>>(buckets, lo, hi);
}

// sum_w 2^(c w) wins[w], Horner from the top window
template <class F>
SIPP_HD Jac<F> combine_windows(const Jac<F>* wins, int W, int c) {
    Jac<F> acc = wins[W - 1];
    for (int w = W - 2; w >= 0; w--) {
        for (int i = 0; i < c; i++) acc = jac_dbl(acc);
        acc = jac_add(acc, wins[w]);
    }
    return acc;
}

// Straus over `nt` terms with their NAF masks (FoldComp.neg unused: the sign is in the term point); digits < 32 * SIPP_FOLD_MASK_WORDS
template <class F>
SIPP_HD Jac<F> straus_terms(const Affine<F>* terms, const FoldComp* naf, size_t nt, int bits) {
    Jac<F> acc = jac_identity<F>();
    for (int i = bits - 1; i >= 0; i--) {
        acc = jac_dbl(acc);
        const uint32_t m = 1u << (i & 31);
        const int w = i >> 5;
        for (size_t t = 0; t < nt; t++) {
            const bool dp = (naf[t].plus[w] & m) != 0, dm = (naf[t].minus[w] & m) != 0;
            if (dp || dm) {
                Affine<F> q = terms[t];
                if (dm) q.y = f_neg(q.y);
                acc = jac_add_affine(acc, q);
            }
        }
    }
    return acc;
}

}  // namespace msm
}  // namespace sipp

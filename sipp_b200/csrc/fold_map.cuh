// fold_map.cuh -- where the batched fold kernels (k_fold.cu, k_wide.cu) find an element: its instance (the index of its FoldPlan),
// its point index i (the fold reads i and i + h, writes i) and its instance's h.  The kernels are templates over the map:
//   UniformFold   the lock-step batch (batch.cu): count instances of h elements each, instance `inst` at points inst * stride
//   RaggedFold    the ragged batch (ragged.cu): a per-round table of the active instances (RaggedInst, launch.h), each with its own
//                 h, found by a binary search over element (or unit) starts
// A wide-fold "unit" is the work of one warp pair of lane groups: two elements of ONE instance when its h is even, one element
// otherwise, so that both groups of a warp run the same digit schedule.
#pragma once
#include <stddef.h>
#include <stdint.h>

#include "launch.h"

namespace sipp {

struct FoldElem {
    size_t inst, i, h;
};

struct UniformFold {
    size_t h, stride, count;
    __device__ __forceinline__ size_t total() const { return count * h; }
    __device__ __forceinline__ FoldElem elem(size_t e) const {
        const size_t inst = e / h;
        return FoldElem{inst, inst * stride + e % h, h};
    }
    // element gi of unit u (gi < 2); valid = false for a shadow (nothing is stored)
    __device__ __forceinline__ FoldElem unit(size_t u, int gi, bool& valid) const {
        const size_t tot = count * h;
        const int epw = (h & 1) ? 1 : 2;
        size_t E = u * epw + (gi % epw);
        valid = E < tot && gi < epw;
        if (E >= tot) E = tot - 1;
        return elem(E);
    }
};

struct RaggedFold {
    const RaggedInst* tab;  // the round's active instances, element and unit starts increasing
    unsigned act;
    size_t elems, units;
    __device__ __forceinline__ size_t total() const { return elems; }
    // last k with start(k) <= x
    template <class Start>
    __device__ __forceinline__ unsigned find(size_t x, Start start) const {
        unsigned lo = 0, hi = act - 1;
        while (lo < hi) {
            const unsigned mid = (lo + hi + 1) >> 1;
            if ((size_t)start(tab[mid]) <= x) lo = mid; else hi = mid - 1;
        }
        return lo;
    }
    __device__ __forceinline__ FoldElem elem(size_t e) const {
        const unsigned k = find(e, [](const RaggedInst& r) { return r.estart; });
        const RaggedInst r = tab[k];
        return FoldElem{k, (size_t)r.base + (e - r.estart), r.h};
    }
    __device__ __forceinline__ FoldElem unit(size_t u, int gi, bool& valid) const {
        valid = u < units;
        if (!valid) u = units - 1;
        const unsigned k = find(u, [](const RaggedInst& r) { return r.ustart; });
        const RaggedInst r = tab[k];
        const int epw = (r.h & 1) ? 1 : 2;
        valid = valid && gi < epw;
        return FoldElem{k, (size_t)r.base + (u - r.ustart) * epw + (gi % epw), r.h};
    }
};

}  // namespace sipp

// tree.cuh -- suffix tree from SA + LCP (SURVEY 8f-5; reference suffix_tree/src/lib.rs:392-505).
//
// The reference inserts the suffixes one by one into a pointer tree.  Its tree is a function of
// the LCP intervals, so every node is found in parallel (DESIGN.md section 6b, row f-5):
//   * boundary j (1 <= j < n, lcp[j] > 0) belongs to the interval [psv[j], nsv[j]) of string
//     depth lcp[j]; the interval's head, its first boundary, is the j with pse[j] == psv[j]
//     (pse = previous smaller-or-equal value);
//   * the reference has no sentinel: when suffix sa[i] is a prefix of suffix sa[i+1]
//     (lcp[i+1] == n - sa[i]), the interval [i, nsv[i+1]) (head i+1) has no node of its own,
//     leaf i takes its place and its children ("absorbed" head);
//   * preorder = (left rank ascending, right end descending), root first.  The nodes with left
//     rank l are the kept heads with psv == l (nested, deeper for smaller j), then leaf l.  So a
//     stable sort by psv of the kept heads listed in descending j puts head p of the sorted list
//     at id 1 + l + p, leaf l at base[l + 1], base[l] = l + (kept heads with psv < l);
//   * parent of interval [l, r): the node of boundary l if lcp[l] >= lcp[r] else of boundary r
//     (lcp[n] = 0); the root if that depth is 0; the absorbing leaf if that node is absorbed.
// The only per-thread walk is from a boundary to its head along pse: the boundaries of one
// node separate children with distinct first bytes, so it takes at most 255 steps.
#pragma once
#include "common.cuh"

namespace b200sa {

constexpr uint32_t TREE_NONE = 0xffffffffu;

struct TreeOut {
    uint32_t *parent, *depth, *lo, *hi, *end, *nchildren;
};

__device__ __forceinline__ bool tree_head(const uint32_t *lcp, const uint32_t *psv, const uint32_t *pse, uint32_t j) {
    return j >= 1 && lcp[j] > 0 && pse[j] == psv[j];
}
// head j whose interval is leaf j-1 (suffix sa[j-1] is a prefix of suffix sa[j])
__device__ __forceinline__ bool tree_absorbed(const uint32_t *sa, const uint32_t *lcp, uint32_t n, uint32_t j) {
    return lcp[j] == n - sa[j - 1];
}

struct TreeIn {
    const uint32_t *sa, *lcp, *psv, *nsv, *pse;
    uint32_t n;
    __device__ __forceinline__ bool head(uint32_t j) const { return tree_head(lcp, psv, pse, j); }
    __device__ __forceinline__ bool absorbed(uint32_t j) const { return tree_absorbed(sa, lcp, n, j); }
    __device__ __forceinline__ bool kept_head(uint32_t j) const { return head(j) && !absorbed(j); }
};

// Kept heads in descending j: element i of the scan is boundary n-1-i.
struct InTreeHead {
    const uint32_t *sa, *lcp, *psv, *pse;
    uint32_t n;
    __device__ uint32_t operator()(uint64_t i) const {
        uint32_t j = n - 1u - (uint32_t)i;
        return tree_head(lcp, psv, pse, j) && !tree_absorbed(sa, lcp, n, j) ? 1u : 0u;
    }
};
struct OutTreeHead {
    const uint32_t *psv;
    uint32_t *key, *val;
    uint32_t n;
    __device__ void operator()(uint64_t i, uint32_t exc, uint32_t v) const {
        if (!v) return;
        uint32_t j = n - 1u - (uint32_t)i;
        key[exc] = psv[j];
        val[exc] = j;
    }
};

// e[l] = one past the last sorted head with left rank l (0 where none)
__global__ void __launch_bounds__(BLK) k_tree_bucket_end(const uint32_t *__restrict__ key, uint32_t m, uint32_t *e) {
    uint32_t p = blockIdx.x * BLK + threadIdx.x;
    if (p >= m) return;
    uint32_t l = key[p];
    if (p + 1 == m || key[p + 1] != l) e[l] = p + 1;
}
// base[l] = l + exclusive max of e (in place over n + 1 entries)
struct OutTreeBase {
    uint32_t *base;
    __device__ void operator()(uint64_t i, uint32_t exc, uint32_t) const { base[i] = (uint32_t)i + exc; }
};

__global__ void __launch_bounds__(BLK) k_tree_internal(TreeIn t, const uint32_t *__restrict__ key,
                                                       const uint32_t *__restrict__ val, uint32_t m,
                                                       const uint32_t *__restrict__ base, uint32_t *headid, TreeOut o) {
    uint32_t p = blockIdx.x * BLK + threadIdx.x;
    if (p >= m) return;
    uint32_t l = key[p], j = val[p], r = t.nsv[j];
    uint32_t u = 1u + l + p;
    headid[j] = u;
    o.lo[u] = l;
    o.hi[u] = r;
    o.depth[u] = t.lcp[j];
    o.end[u] = 1u + base[r];
}

__device__ __forceinline__ uint32_t tree_parent(const TreeIn &t, const uint32_t *__restrict__ base,
                                                const uint32_t *__restrict__ headid, uint32_t l, uint32_t r) {
    uint32_t a = t.lcp[l], b = r < t.n ? t.lcp[r] : 0u;
    uint32_t h = a >= b ? l : r;
    if ((a >= b ? a : b) == 0) return 0u;
    while (t.pse[h] != t.psv[h]) h = t.pse[h];
    return t.absorbed(h) ? base[t.psv[h] + 1] : headid[h];
}

// Thread i: leaf i, and boundary i when it heads a node; parents and child counts
// (o.nchildren zeroed beforehand; a node has at most 256 children).
__global__ void __launch_bounds__(BLK) k_tree_link(TreeIn t, const uint32_t *__restrict__ base,
                                                   const uint32_t *__restrict__ headid, TreeOut o) {
    uint32_t i = blockIdx.x * BLK + threadIdx.x;
    if (i >= t.n) return;
    uint32_t u = base[i + 1];
    bool absorbing = i + 1 < t.n && t.head(i + 1) && t.absorbed(i + 1);
    uint32_t r = absorbing ? t.nsv[i + 1] : i + 1;
    uint32_t par = tree_parent(t, base, headid, i, r);
    o.lo[u] = i;
    o.hi[u] = r;
    o.depth[u] = t.n - t.sa[i];
    o.end[u] = 1u + base[r];
    o.parent[u] = par;
    atomicAdd(o.nchildren + par, 1u);
    if (t.kept_head(i)) {
        uint32_t v = headid[i];
        uint32_t pv = tree_parent(t, base, headid, t.psv[i], t.nsv[i]);
        o.parent[v] = pv;
        atomicAdd(o.nchildren + pv, 1u);
    }
    if (i == 0) {
        o.parent[0] = TREE_NONE;
        o.depth[0] = 0u;
        o.lo[0] = 0u;
        o.hi[0] = t.n;
        o.end[0] = 1u + base[t.n];
    }
}

}  // namespace b200sa

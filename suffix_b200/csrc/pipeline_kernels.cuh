// pipeline_kernels.cuh -- functors and small kernels for the glue phases:
//   K3  LMS grouping by first byte            (reference P5,  src/table.rs:411-416)
//   K6  compaction of sorted LMS substrings   (reference P10, src/table.rs:450-463)
//   K7  naming by neighbour equality          (reference P11, src/table.rs:465-482, wstring_equal :802-820)
//   K8  reduced string in text order          (reference P12, src/table.rs:484-492)
//   K9  base case (unique names)              (reference P13, src/table.rs:501-506) -- no kernel needed
//   K10 un-rename ranks -> text positions     (reference P15-P16, src/table.rs:512-530)
//   k-gram sort + rank-pair doubling on the reduced string (stands in for the recursion at src/table.rs:499)
//   K12/K13 LCP: direct per-pair fast path, Phi / two-level PLCP linear path (reference semantics src/table.rs:348-361)
//   batched positions()                       (reference src/table.rs:223-259)
#pragma once
#include "classify.cuh"

namespace b200sa {

// ------------------------------------------------------------ scan functors
struct InPopcWords {            // popcount of bitmap words
    const uint32_t *bm;
    __device__ uint32_t operator()(uint64_t i) const { return __popc(bm[i]); }
};
struct OutStoreExcl {           // out[i] = exclusive prefix
    uint32_t *out;
    __device__ void operator()(uint64_t i, uint32_t exc, uint32_t) const { out[i] = exc; }
};
struct InArray {
    const uint32_t *a;
    __device__ uint32_t operator()(uint64_t i) const { return a[i]; }
};

// K6: keep SA entries that are LMS positions
struct InIsLmsEntry {
    const uint32_t *sa; const uint32_t *lmsb;
    __device__ uint32_t operator()(uint64_t i) const { return bit_at(lmsb, sa[i]); }
};
struct OutCompactSa {
    const uint32_t *sa; uint32_t *out;
    __device__ void operator()(uint64_t i, uint32_t exc, uint32_t v) const { if (v) out[exc] = sa[i]; }
};

// ------------------------------------------------------------ K3 functors
struct DigTextAtPos {           // digit = first byte of the LMS suffix
    const uint8_t *text; const uint32_t *pos;
    __device__ uint32_t operator()(uint64_t i) const { return __ldg(text + pos[i]); }
};
struct MoveU32 {
    const uint32_t *in; uint32_t *out;
    __device__ void operator()(uint64_t i, uint32_t dst) const { out[dst] = in[i]; }
};

// ------------------------------------------------------------ K7 naming
// LMS-substring equality with the reference's semantics (src/table.rs:802-820):
// equal chars and equal type class position by position; equal once a later
// position of either is a Valley; running off the text means different.
// Two LMS substrings are equal iff they have the same length and the same
// chars: the types of positions i..j-1 of a substring T[i..j] are determined by
// its chars (T[j-1] > T[j] because j-1 is L and j is S), the first and last
// positions are Valleys in both, and a length mismatch shows up in the
// reference as a type mismatch at the shorter one's last position.  A substring
// that runs off the text (no later Valley) equals nothing (:814-819).
// flag[i] = 1 iff sorted LMS substring i starts a new name.  Substrings longer
// than NAME_SOLO chars (runs: poly-N, padding) are finished warp-cooperatively.
constexpr uint32_t NAME_SOLO = 256;
template <int BITS>
__global__ void __launch_bounds__(BLK) k_name_flags(const void *__restrict__ ptext, uint32_t n,
                                                    const uint32_t *__restrict__ lmsb,
                                                    const uint32_t *__restrict__ sorted, uint32_t m, uint8_t *flag) {
    uint32_t i = blockIdx.x * BLK + threadIdx.x;
    bool live = i < m;
    uint32_t a = 0, b = 0, len = 0;      // len = chars to compare (0: already decided)
    uint8_t f = 1;
    if (live && i > 0) {
        a = sorted[i]; b = sorted[i - 1];
        uint32_t la = next_lms_dist(lmsb, n, a);
        if (la != 0 && la == next_lms_dist(lmsb, n, b)) len = la + 1;
    }
    uint32_t solo = len < NAME_SOLO ? len : NAME_SOLO;
    uint32_t got = len ? text_match<BITS>(ptext, a, b, solo) : 0u;
    uint32_t pending = __ballot_sync(FULL, len > NAME_SOLO && got == NAME_SOLO);
    while (pending) {
        int src = __ffs(pending) - 1;
        pending &= pending - 1;
        uint32_t aa = __shfl_sync(FULL, a, src) + NAME_SOLO, bb = __shfl_sync(FULL, b, src) + NAME_SOLO;
        uint32_t ll = __shfl_sync(FULL, len, src) - NAME_SOLO;
        uint32_t more = text_match_warp<BITS>(ptext, aa, bb, ll);
        if ((int)lane_id() == src) got += more;
    }
    if (len && got == len) f = 0;
    if (live) flag[i] = f;
}
struct InFlagU8 {
    const uint8_t *f;
    __device__ uint32_t operator()(uint64_t i) const { return f[i]; }
};
// K8: reduced[text_rank(sorted[i])] = name(i) = inclusive(flag) - 1
struct OutReduced {
    const uint32_t *sorted; const uint32_t *lmsb; const uint32_t *lmsrank; uint32_t *reduced;
    __device__ void operator()(uint64_t i, uint32_t exc, uint32_t v) const {
        reduced[lms_text_rank(lmsb, lmsrank, sorted[i])] = exc + v - 1u;
    }
};

// Doubling start-up straight from the sorted LMS substrings (no re-sort of the
// names): slot i of the reduced SA holds text_rank(sorted[i]); its group is the
// run of equal names it sits in; rank[] plays the role of the reduced string
// (reference P11-P12, src/table.rs:465-492, kept as ranks instead of names).
struct InFlagPos {
    const uint8_t *f;
    __device__ uint32_t operator()(uint64_t i) const { return f[i] ? (uint32_t)i : 0u; }
};
struct OutInitFromSorted {
    const uint32_t *sorted; const uint32_t *lmsb; const uint32_t *lmsrank; const uint8_t *flag; uint32_t m; int write_all;
    uint32_t *sa_r; uint32_t *grp; uint32_t *rank;
    __device__ void operator()(uint64_t i, uint32_t exc, uint32_t v) const {
        uint32_t g = exc > v ? exc : v;
        uint32_t tr = lms_text_rank(lmsb, lmsrank, sorted[i]);
        sa_r[i] = tr;
        grp[i] = g;
        // members of larger groups get their rank from the first refinement round,
        // which sorts all of them; only name-singletons need it now (saves the
        // random scatter for ~98 % of a DNA-like reduced string)
        bool single = flag[i] && (i + 1 == m || flag[i + 1]);
        if (single || write_all) rank[tr] = g + 1u;
    }
};
// K9 (all names unique): the sorted LMS substrings already are the reduced SA -- OutInitFromSorted
// writes sa_r[i] = text_rank(sorted[i]); no inversion kernel is needed (reference :501-506).
// K10: sorted LMS suffixes = lmspos[sa_r[i]]
__global__ void __launch_bounds__(BLK) k_unrename(const uint32_t *sa_r, const uint32_t *lmspos, uint32_t m,
                                                  uint32_t *out) {
    uint32_t i = blockIdx.x * BLK + threadIdx.x;
    if (i < m) out[i] = lmspos[sa_r[i]];
}

// ------------------------------------------------------------ doubling
__global__ void __launch_bounds__(BLK) k_iota(uint32_t *a, uint32_t m) {
    uint32_t i = blockIdx.x * BLK + threadIdx.x;
    if (i < m) a[i] = i;
}
// Round-0 key of k consecutive symbols: sym+1 per slot (0 = beyond the end, so
// a proper prefix sorts first), bw bits per slot, first symbol most significant.
template <class K>
__global__ void __launch_bounds__(BLK) k_multi_key(const uint32_t *__restrict__ R, uint32_t m, uint32_t k,
                                                   uint32_t bw, K *keys) {
    uint32_t i = blockIdx.x * BLK + threadIdx.x;
    if (i >= m) return;
    K key = 0;
    for (uint32_t j = 0; j < k; j++) {
        uint64_t p = (uint64_t)i + j;
        K v = p < m ? (K)(__ldg(R + p) + 1u) : (K)0;
        key = (key << bw) | v;
    }
    keys[i] = key;
}
// Same key for a list of suffixes (first refinement round: jumps from depth 1
// to depth k in one sort).
template <class K>
__global__ void __launch_bounds__(BLK) k_multi_key_list(const uint32_t *__restrict__ R, uint32_t m,
                                                        const uint32_t *__restrict__ suf, uint32_t na, uint32_t k,
                                                        uint32_t bw, K *keys) {
    uint32_t idx = blockIdx.x * BLK + threadIdx.x;
    if (idx >= na) return;
    uint32_t i = suf[idx];
    K key = 0;
    for (uint32_t j = 0; j < k; j++) {
        uint64_t p = (uint64_t)i + j;
        K v = p < m ? (K)(__ldg(R + p) + 1u) : (K)0;
        key = (key << bw) | v;
    }
    keys[idx] = key;
}
template <class K>
struct DigKey {
    const K *keys; uint32_t shift;
    __device__ uint32_t operator()(uint64_t i) const { return (uint32_t)(keys[i] >> shift) & 0xffu; }
};
template <class K>
struct MoveKV {
    const K *kin; const uint32_t *vin; K *kout; uint32_t *vout;
    __device__ void operator()(uint64_t i, uint32_t dst) const { kout[dst] = kin[i]; vout[dst] = vin[i]; }
};
// group-start scan input: (key differs from predecessor) ? position id : 0
// pos == nullptr -> the position id is the index itself.
template <class K>
struct InGroupStart {
    const K *keys; const uint32_t *pos;
    __device__ uint32_t operator()(uint64_t i) const {
        bool head = (i == 0) || (keys[i] != keys[i - 1]);
        return head ? (pos ? pos[i] : (uint32_t)i) : 0u;
    }
};
// consumes the inclusive max-scan: grp[i] = start slot of i's group,
// rank[suffix] = grp + 1, and (optionally) sa_r[slot] = suffix.
struct OutGroupRank {
    const uint32_t *suf; const uint32_t *pos; uint32_t *grp; uint32_t *rank; uint32_t *sa_r;
    __device__ void operator()(uint64_t i, uint32_t exc, uint32_t v) const {
        uint32_t g = exc > v ? exc : v;
        grp[i] = g;
        uint32_t s = suf[i];
        rank[s] = g + 1u;
        if (sa_r) sa_r[pos ? pos[i] : (uint32_t)i] = s;
    }
};
// active = member of a group with more than one element
template <class K>
struct InActive {
    const K *keys; uint64_t cnt;
    __device__ uint32_t operator()(uint64_t i) const {
        bool head = (i == 0) || (keys[i] != keys[i - 1]);
        bool tail = (i + 1 == cnt) || (keys[i + 1] != keys[i]);
        return (head && tail) ? 0u : 1u;
    }
};
// Fused per-round pass: one (max, sum) pair scan derives the group start of every
// sorted element AND compacts the still-ambiguous ones (the two used to be separate
// scans, each reading the keys twice).
template <class K>
struct InGroupActive {
    const K *keys; const uint32_t *pos; uint64_t cnt;
    __device__ unsigned long long operator()(uint64_t i) const {
        bool head = (i == 0) || (keys[i] != keys[i - 1]);
        bool tail = (i + 1 == cnt) || (keys[i + 1] != keys[i]);
        uint32_t hi = head ? (pos ? pos[i] : (uint32_t)i) : 0u;
        uint32_t lo = (head && tail) ? 0u : 1u;
        return ((unsigned long long)hi << 32) | lo;
    }
};
struct OutGroupRankCompact {
    const uint32_t *suf; const uint32_t *pos; uint32_t *rank; uint32_t *sa_r;
    uint32_t *opos; uint32_t *osuf; uint32_t *ogrp;
    __device__ void operator()(uint64_t i, unsigned long long exc, unsigned long long v) const {
        uint32_t eh = (uint32_t)(exc >> 32), vh = (uint32_t)(v >> 32);
        uint32_t g = eh > vh ? eh : vh;
        uint32_t s = suf[i];
        uint32_t p = pos ? pos[i] : (uint32_t)i;
        rank[s] = g + 1u;
        if (sa_r) sa_r[p] = s;
        if ((uint32_t)v) {                      // member of a group that is still ambiguous
            uint32_t k = (uint32_t)exc;
            opos[k] = p; osuf[k] = s; ogrp[k] = g;
        }
    }
};
struct OutCompactActive {
    const uint32_t *pos; const uint32_t *suf; const uint32_t *grp;   // pos==nullptr -> index
    uint32_t *opos; uint32_t *osuf; uint32_t *ogrp;
    __device__ void operator()(uint64_t i, uint32_t exc, uint32_t v) const {
        if (v) { opos[exc] = pos ? pos[i] : (uint32_t)i; osuf[exc] = suf[i]; ogrp[exc] = grp[i]; }
    }
};
// key = (group start << b2) | rank[suffix + h]   (0 beyond the end: a proper
// prefix sorts first, matching slice `cmp`, src/table.rs:374)
__global__ void __launch_bounds__(BLK) k_pair_keys(const uint32_t *agrp, const uint32_t *asuf, const uint32_t *rank,
                                                   uint32_t na, uint32_t m, uint32_t h, uint32_t b2, uint64_t *keys) {
    uint32_t k = blockIdx.x * BLK + threadIdx.x;
    if (k >= na) return;
    uint64_t s2 = (uint64_t)asuf[k] + h;
    uint32_t r2 = s2 < m ? rank[s2] : 0u;
    keys[k] = ((uint64_t)agrp[k] << b2) | r2;
}

// Later refinement rounds: after the k-gram round almost every ambiguous group
// has 2-3 members, so a global radix sort (7 passes) is overkill.  Each element
// finds its group (run of equal high key part) by scanning its neighbours and
// takes the rank of its key inside the group by counting -- O(g) reads, one
// scatter.  Groups larger than GL_LIMIT raise *overflow and the caller falls
// back to the one-sweep sort for that round.
// Probe: group sizes (capped at 128) of ~4096 evenly spaced elements; stats[0] =
// how many of them sit in groups of >= 128.  The host skips the local sort when
// such groups are common (each of their members would scan the whole group).
__global__ void __launch_bounds__(BLK) k_group_probe(const uint64_t *__restrict__ keys, uint32_t na, uint32_t b2,
                                                     uint32_t stride, uint32_t *stats) {
    uint64_t kk = (uint64_t)(blockIdx.x * BLK + threadIdx.x) * stride;
    if (kk >= na) return;
    uint32_t k = (uint32_t)kk;
    const uint64_t g = keys[k] >> b2;
    uint32_t lo = k, hi = k + 1, size = 1;
    while (lo > 0 && size < 128u && (keys[lo - 1] >> b2) == g) { lo--; size++; }
    while (hi < na && size < 128u && (keys[hi] >> b2) == g) { hi++; size++; }
    if (size >= 128u) atomicAdd(&stats[0], 1u);      // member of a group of >= 128
    atomicMax(&stats[1], size);
}
constexpr int GL_LIMIT = 1024;
__global__ void __launch_bounds__(BLK) k_group_local_sort(const uint64_t *__restrict__ keys,
                                                          const uint32_t *__restrict__ suf, uint32_t na, uint32_t b2,
                                                          uint64_t *kout, uint32_t *sout, uint32_t *overflow) {
    uint32_t k = blockIdx.x * BLK + threadIdx.x;
    if (k >= na) return;
    const uint64_t mine = keys[k];
    const uint64_t g = mine >> b2;
    uint32_t lo = k, hi = k + 1;
    int steps = 0;
    while (lo > 0 && (keys[lo - 1] >> b2) == g) {
        lo--;
        if (++steps > GL_LIMIT) { *overflow = 1u; return; }
    }
    while (hi < na && (keys[hi] >> b2) == g) {
        hi++;
        if (++steps > GL_LIMIT) { *overflow = 1u; return; }
    }
    uint32_t pos = 0;
    for (uint32_t j = lo; j < hi; j++) {
        uint64_t o = keys[j];
        pos += (o < mine || (o == mine && j < k)) ? 1u : 0u;
    }
    kout[lo + pos] = mine;
    sout[lo + pos] = suf[k];
}

// ------------------------------------------------------------ LCP
// Phi / PLCP formulation of Kasai (same values as the reference's
// lcp_lens_quadratic, src/table.rs:348-361; the algorithm is the byte-level
// version of the commented-out lcp_lens_linear, :314-346):
//   phi[sa[r]] = sa[r-1]            (one random write per suffix)
//   plcp[i]    = lcp(i, phi[i])     (text order; plcp[i] >= plcp[i-1]-1)
//   lcp[r]     = plcp[sa[r]]        (one random read per suffix)
// Fast path: the reference's own definition, lcp_len(suffix sa[r-1], suffix sa[r])
// (src/table.rs:356-365), evaluated directly per adjacent pair with word-wide
// compares on the (L2-resident) packed text, capped at `cap` chars.  Pairs that
// reach the cap are counted; if any exist the caller recomputes everything with
// the linear Phi/PLCP path below (the direct form is quadratic on repetitive text).
template <int BITS, int K = 1>
__global__ void __launch_bounds__(BLK) k_lcp_direct(const void *__restrict__ ptext, uint32_t n,
                                                    const uint32_t *__restrict__ sa, uint32_t *lcp, uint32_t cap,
                                                    uint32_t *capped) {
    if (BITS == 8) {
        uint32_t r = blockIdx.x * BLK + threadIdx.x;
        const bool live = r < n;
        uint32_t h = 0, room = 0;
        if (live && r > 0) {
            uint32_t a = sa[r - 1], b = sa[r];
            room = n - (a > b ? a : b);
            uint32_t limit = room < cap ? room : cap;
            h = text_match<BITS>(ptext, a, b, limit);
        }
        if (live) {
            lcp[r] = h;
            if (r > 0 && h == cap && room > cap) atomicAdd(capped, 1u);
        }
    } else {
        // Packed text: the first window of suffix sa[r] serves the pairs (r-1, r) AND (r, r+1): every lane
        // loads its own window once and takes its left neighbour's from the lane below (lane 0 loads
        // both) -- the kernel is bound by the number of divergent window loads, and this halves them.
        // A warp owns K runs of 32 consecutive ranks; the K window gathers of a lane are in flight together.
        constexpr int PB = (BITS == 8 ? 4 : BITS);
        constexpr uint32_t CPW = 32 / PB;
        const uint32_t wbase = (blockIdx.x * BLK + (threadIdx.x & ~31u)) * (uint32_t)K + lane_id();
        uint32_t b[K], xb[K];
        bool live[K];
#pragma unroll
        for (int k = 0; k < K; k++) {
            uint32_t r = wbase + 32u * k;
            live[k] = r < n;
            b[k] = live[k] ? sa[r] : 0u;
        }
#pragma unroll
        for (int k = 0; k < K; k++) xb[k] = live[k] ? text_bits<PB>(ptext, b[k]) : 0u;
#pragma unroll
        for (int k = 0; k < K; k++) {
            uint32_t r = wbase + 32u * k;
            uint32_t a = __shfl_up_sync(FULL, b[k], 1), xa = __shfl_up_sync(FULL, xb[k], 1);
            uint32_t pa = 0, pxa = 0;
            if (k > 0) { pa = __shfl_sync(FULL, b[k > 0 ? k - 1 : 0], 31); pxa = __shfl_sync(FULL, xb[k > 0 ? k - 1 : 0], 31); }
            if (lane_id() == 0) {                       // left neighbour of the run's first rank
                if (k > 0) { a = pa; xa = pxa; }
                else if (live[k] && r > 0) { a = sa[r - 1]; xa = text_bits<PB>(ptext, a); }
            }
            uint32_t h = 0, room = 0;
            if (live[k] && r > 0) {
                room = n - (a > b[k] ? a : b[k]);
                uint32_t limit = room < cap ? room : cap;
                uint32_t x = xa ^ xb[k];
                uint32_t first = x ? (uint32_t)(__ffs(x) - 1) / PB : CPW;       // equal leading chars inside the window
                if (first < CPW || limit <= CPW) h = first < limit ? first : limit;
                else h = CPW + text_match<BITS>(ptext, a + CPW, b[k] + CPW, limit - CPW);
            }
            if (live[k]) {
                lcp[r] = h;
                if (r > 0 && h == cap && room > cap) atomicAdd(capped, 1u);
            }
        }
    }
}

// lcp-only entry points: the caller's table must be a permutation of 0..n-1 (every LCP
// kernel indexes text / phi with sa[r]).  *bad counts out-of-range and repeated entries.
__global__ void __launch_bounds__(BLK) k_sa_validate(const uint32_t *__restrict__ sa, uint32_t n, uint32_t *seen,
                                                     uint32_t *bad) {
    // fire-and-forget reductions (RED, no return value) into the bitmap: a repeated entry shows up as a
    // missing bit, which k_sa_validate_count finds (n entries < n without repeats <=> n bits set)
    uint32_t r0 = (blockIdx.x * BLK + threadIdx.x) * 4u;
    uint32_t wrong = 0;
    if (r0 + 4u <= n && (reinterpret_cast<uintptr_t>(sa) & 15) == 0) {
        uint4 v = *reinterpret_cast<const uint4 *>(sa + r0);
        uint32_t s[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int q = 0; q < 4; q++) {
            if (s[q] >= n) wrong++;
            else atomicOr(&seen[s[q] >> 5], 1u << (s[q] & 31));
        }
    } else {
        for (uint32_t r = r0; r < n && r < r0 + 4u; r++) {
            uint32_t s = sa[r];
            if (s >= n) wrong++;
            else atomicOr(&seen[s >> 5], 1u << (s & 31));
        }
    }
    if (wrong) atomicAdd(bad, wrong);
}
// bad += 1 unless exactly n bits are set in seen[0 .. ceil(n/32))
__global__ void __launch_bounds__(BLK) k_sa_validate_count(const uint32_t *__restrict__ seen, uint32_t n, uint32_t *cnt) {
    uint32_t nw = (n + 31u) / 32u, c = 0;
    for (uint32_t i = blockIdx.x * BLK + threadIdx.x; i < nw; i += gridDim.x * BLK) c += __popc(seen[i]);
    c = __reduce_add_sync(FULL, c);
    if (lane_id() == 0 && c) atomicAdd(cnt, c);
}
__global__ void k_sa_validate_verdict(const uint32_t *cnt, uint32_t n, uint32_t *bad) {
    if (*cnt != n) atomicAdd(bad, 1u);
}
// Is a permutation (checked by k_sa_validate first) THE suffix array of the text?  The Phi / PLCP
// path below is Kasai's algorithm: it relies on plcp[i] >= plcp[i-1] - 1, which only holds for the
// sorted table.  Neighbour-order test with the inverse: for every adjacent pair (a, b) =
// (sa[r-1], sa[r]), T[a] < T[b], or T[a] == T[b] and suffix a+1 precedes suffix b+1 (the empty
// suffix precedes all).  *bad is set if any pair is out of order.
__global__ void __launch_bounds__(BLK) k_sa_inverse(const uint32_t *__restrict__ sa, uint32_t n, uint32_t *inv) {
    uint32_t r = blockIdx.x * BLK + threadIdx.x;
    if (r < n) inv[sa[r]] = r;
}
__global__ void __launch_bounds__(BLK) k_sa_sorted(const uint8_t *__restrict__ text, uint32_t n,
                                                   const uint32_t *__restrict__ sa, const uint32_t *__restrict__ inv,
                                                   uint32_t *bad) {
    uint32_t r = blockIdx.x * BLK + threadIdx.x;
    bool wrong = false;
    if (r > 0 && r < n) {
        uint32_t a = sa[r - 1], b = sa[r];
        uint32_t ca = __ldg(text + a), cb = __ldg(text + b);
        if (ca != cb) wrong = ca > cb;
        else if (a + 1 == n) wrong = false;          // "c" precedes "c..."
        else if (b + 1 == n) wrong = true;
        else wrong = inv[a + 1] >= inv[b + 1];
    }
    if (__ballot_sync(FULL, wrong) && lane_id() == 0) atomicOr(bad, 1u);
}

constexpr uint32_t PHI_NONE = 0xffffffffu;
__global__ void __launch_bounds__(BLK) k_phi(const uint32_t *__restrict__ sa, uint32_t n, uint32_t *phi) {
    uint32_t r = blockIdx.x * BLK + threadIdx.x;
    if (r < n) phi[sa[r]] = r ? sa[r - 1] : PHI_NONE;
}
// Binned variant: the (position, predecessor) pairs are first partitioned by the
// top 8 bits of the position (one one-sweep pass), so that the scatter below
// walks the phi array window by window and every 32-byte sector is completed in
// L2 before it is written back (no read-modify-write of partial sectors).
struct LoadPhiPrev {
    const uint32_t *sa;
    __device__ __forceinline__ uint32_t operator()(uint64_t r) const { return r ? sa[r - 1] : PHI_NONE; }
};
__global__ void __launch_bounds__(BLK) k_phi_apply(const uint32_t *__restrict__ pos, const uint32_t *__restrict__ prev,
                                                   uint32_t n, uint32_t *phi) {
    uint32_t i = blockIdx.x * BLK + threadIdx.x;
    if (i < n) phi[pos[i]] = prev[i];
}
// One thread owns LCP_CHUNK consecutive text positions: the first starts from
// h = 0, the rest reuse h-1.  buf holds phi on entry and plcp on exit.
constexpr int LCP_CHUNK = 32;
// Level 1: exact plcp at every LCP_CHUNK-th text position.  One thread walks 32
// consecutive samples with the carry plcp[i+32] >= plcp[i]-32, so a restart from
// h = 0 happens once per 1024 positions instead of once per 32 (inside a run or
// repeat of length L a restart costs O(L)).
constexpr uint32_t LCP_SOLO = 256;       // chars a lane compares alone before the warp takes over
// (t_off, pos_end): text-range sharding (multi-GPU LCP) -- threads start at sample group t_off and
// positions at or beyond pos_end belong to another rank.
template <int BITS>
__global__ void __launch_bounds__(BLK) k_plcp_samples(const void *__restrict__ ptext, uint32_t n,
                                                      const uint32_t *__restrict__ phi, uint32_t *samp,
                                                      uint64_t t_off, uint64_t pos_end) {
    uint64_t t = t_off + (uint64_t)blockIdx.x * BLK + threadIdx.x;
    uint64_t s0 = t * 32;
    uint32_t h = 0;
    for (int j = 0; j < 32; j++) {                       // no early exit: the warp cooperates below
        uint64_t sidx = s0 + j, i = sidx * LCP_CHUNK;
        bool live = i < n && i < pos_end;
        uint32_t jp = live ? phi[i] : PHI_NONE;
        bool cmp = live && jp != PHI_NONE;
        uint32_t a = 0, b = 0, limit = 0, got = 0;
        if (cmp) {
            a = (uint32_t)i + h; b = jp + h;
            limit = n - (a > b ? a : b);
            uint32_t solo = limit < LCP_SOLO ? limit : LCP_SOLO;
            got = text_match<BITS>(ptext, a, b, solo);
        }
        // lanes whose match ran through the solo window: finish them one by one, warp-wide
        uint32_t pending = __ballot_sync(FULL, cmp && got == LCP_SOLO && limit > LCP_SOLO);
        while (pending) {
            int src = __ffs(pending) - 1;
            pending &= pending - 1;
            uint32_t aa = __shfl_sync(FULL, a, src) + LCP_SOLO, bb = __shfl_sync(FULL, b, src) + LCP_SOLO;
            uint32_t ll = __shfl_sync(FULL, limit, src) - LCP_SOLO;
            uint32_t more = text_match_warp<BITS>(ptext, aa, bb, ll);
            if ((int)lane_id() == src) got += more;
        }
        if (live) {
            h = cmp ? h + got : 0u;
            samp[sidx] = h;
            h = h > (uint32_t)LCP_CHUNK ? h - LCP_CHUNK : 0u;
        }
    }
}
// Level 2: every thread owns LCP_CHUNK consecutive positions; the first one takes
// its value from the samples, the rest reuse h-1.  buf holds phi on entry and plcp
// on exit.
template <int BITS>
__global__ void __launch_bounds__(BLK) k_plcp(const void *__restrict__ ptext, uint32_t n, uint32_t *buf,
                                              const uint32_t *__restrict__ samp, uint64_t t_off, uint64_t pos_end) {
    uint64_t t = t_off + (uint64_t)blockIdx.x * BLK + threadIdx.x;
    uint64_t i0 = t * LCP_CHUNK;
    if (i0 >= n || i0 >= pos_end) return;
    uint64_t i1 = i0 + LCP_CHUNK;
    if (i1 > n) i1 = n;
    uint32_t h = samp[t];
    buf[i0] = h;
    if (h > 0) h--;
    for (uint64_t i = i0 + 1; i < i1; i++) {
        uint32_t j = buf[i];
        if (j == PHI_NONE) { buf[i] = 0; h = 0; continue; }
        uint32_t a = (uint32_t)i + h, b = j + h;     // a, b <= n: h never exceeds the shorter suffix on a
                                                     // sorted table (k_sa_sorted checks caller tables)
        uint32_t limit = n - (a > b ? a : b);
        h += text_match<BITS>(ptext, a, b, limit);
        buf[i] = h;
        if (h > 0) h--;
    }
}
// phi restricted to the text range [lo, hi) of one rank (the whole SA is scanned; the writes fall
// into a range small enough to stay in L2)
__global__ void __launch_bounds__(BLK) k_phi_range(const uint32_t *__restrict__ sa, uint32_t n, uint32_t lo, uint32_t hi,
                                                   uint32_t *phi) {
    uint32_t r = blockIdx.x * BLK + threadIdx.x;
    if (r >= n) return;
    uint32_t i = sa[r];
    if (i >= lo && i < hi) phi[i] = r ? sa[r - 1] : PHI_NONE;
}
__global__ void __launch_bounds__(BLK) k_lcp_gather_range(const uint32_t *__restrict__ sa, const uint32_t *__restrict__ plcp,
                                                          uint32_t lo, uint32_t hi, uint32_t *out) {
    uint32_t r = lo + blockIdx.x * BLK + threadIdx.x;
    if (r < hi) out[r - lo] = plcp[sa[r]];
}
__global__ void __launch_bounds__(BLK) k_lcp_gather(const uint32_t *__restrict__ sa, const uint32_t *__restrict__ plcp,
                                                    uint32_t n, uint32_t *lcp) {
    uint32_t r = blockIdx.x * BLK + threadIdx.x;
    if (r < n) lcp[r] = plcp[sa[r]];
}

// ------------------------------------------------------------ batched positions
__device__ __forceinline__ int cmp_query_suffix(const uint8_t *__restrict__ text, uint32_t n, uint32_t s,
                                                const uint8_t *__restrict__ q, uint32_t m, bool *is_prefix) {
    // compares query with text[s..]; *is_prefix = suffix starts with query
    uint32_t ls = n - s, l = ls < m ? ls : m, k = 0;
    while (k < l) {
        uint32_t a = q[k], b = __ldg(text + s + k);
        if (a != b) { *is_prefix = false; return a < b ? -1 : 1; }
        k++;
    }
    *is_prefix = (m <= ls);
    return (m <= ls) ? (m == ls ? 0 : -1) : 1;
}
// One thread per query: reference early-outs (src/table.rs:228-235), then the
// two binary searches (:244-250).
__global__ void __launch_bounds__(BLK) k_positions(const uint8_t *__restrict__ text, uint32_t n,
                                                   const uint32_t *__restrict__ sa, const uint8_t *__restrict__ qs,
                                                   const uint64_t *__restrict__ qoff, uint32_t nq,
                                                   uint32_t *out_start, uint32_t *out_end) {
    uint32_t qi = blockIdx.x * BLK + threadIdx.x;
    if (qi >= nq) return;
    const uint8_t *q = qs + qoff[qi];
    uint32_t m = (uint32_t)(qoff[qi + 1] - qoff[qi]);
    uint32_t start = 0, end = 0;
    if (n > 0 && m > 0) {
        bool pre;
        int c0 = cmp_query_suffix(text, n, sa[0], q, m, &pre);
        bool out = (c0 < 0 && !pre);
        if (!out) { bool p2; out = cmp_query_suffix(text, n, sa[n - 1], q, m, &p2) > 0; }
        if (!out) {
            uint32_t lo = 0, hi = n;
            while (lo < hi) {                               // first suffix >= query
                uint32_t mid = lo + (hi - lo) / 2;
                bool p;
                int c = cmp_query_suffix(text, n, sa[mid], q, m, &p);
                if (c <= 0) hi = mid; else lo = mid + 1;
            }
            start = lo;
            uint32_t lo2 = 0, hi2 = n - start;
            while (lo2 < hi2) {                             // first suffix not starting with query
                uint32_t mid = lo2 + (hi2 - lo2) / 2;
                bool p;
                cmp_query_suffix(text, n, sa[start + mid], q, m, &p);
                if (!p) hi2 = mid; else lo2 = mid + 1;
            }
            end = start + lo2;
        }
    }
    out_start[qi] = start;
    out_end[qi] = end;
}

// ------------------------------------------------------------ generalized suffix array (SURVEY 8f-3)
// document of a text position: doc_starts[d] <= pos < doc_starts[d+1] (ascending, doc_starts[ndocs] = n);
// positions of separator bytes map to the document they terminate.
__global__ void __launch_bounds__(BLK) k_doc_ids(const uint32_t *__restrict__ pos, uint64_t count,
                                                 const uint32_t *__restrict__ doc_starts, uint32_t ndocs,
                                                 uint32_t *doc, uint32_t *off) {
    uint64_t i = (uint64_t)blockIdx.x * BLK + threadIdx.x;
    if (i >= count) return;
    uint32_t p = pos[i], lo = 0, hi = ndocs;            // last d with doc_starts[d] <= p
    while (hi - lo > 1) {
        uint32_t mid = lo + (hi - lo) / 2;
        if (__ldg(doc_starts + mid) <= p) lo = mid; else hi = mid;
    }
    doc[i] = lo;
    off[i] = p - __ldg(doc_starts + lo);
}

// ------------------------------------------------------------ LCP-interval tree (SURVEY 8f-4)
// The internal nodes of the suffix tree are the LCP intervals (reference builds the pointer tree
// serially from SA + LCP, suffix_tree/src/lib.rs:392-505).  For every rank i: psv[i] = largest j < i
// with lcp[j] < lcp[i] (NONE if none), nsv[i] = smallest j > i with lcp[j] < lcp[i] (n if none): the
// node that owns boundary i is the interval [psv[i], nsv[i]) of string depth lcp[i].  Minima over
// blocks of 32^k entries let every thread skip whole blocks.
constexpr uint32_t ANSV_NONE = 0xffffffffu;
__global__ void __launch_bounds__(BLK) k_min32(const uint32_t *__restrict__ in, uint64_t n_in, uint32_t *out) {
    uint64_t b = (uint64_t)blockIdx.x * BLK + threadIdx.x;
    uint64_t i0 = b * 32;
    if (i0 >= n_in) return;
    uint32_t m = 0xffffffffu;
    for (int k = 0; k < 32 && i0 + k < n_in; k++) { uint32_t v = in[i0 + k]; m = v < m ? v : m; }
    out[b] = m;
}
struct AnsvLevels {
    const uint32_t *lv[8];     // lv[0] = lcp, lv[k] = minima over 32^k entries
    uint64_t cnt[8];
    int nlev;
};
// STRICT: nearest value < v; otherwise nearest value <= v (block minima serve both).
template <bool STRICT>
__device__ __forceinline__ bool ansv_hit(uint32_t x, uint32_t v) { return STRICT ? x < v : x <= v; }
template <bool STRICT>
__device__ __forceinline__ uint32_t ansv_left(const AnsvLevels &L, uint64_t i, uint32_t v) {
    // climb: at level k, scan the siblings to the left inside the parent block; a block with min < v holds the answer
    uint64_t idx = i;
    int k = 0;
    while (true) {
        uint64_t first = idx & ~(uint64_t)31;
        uint64_t j = idx;
        bool found = false;
        while (j > first) {
            j--;
            if (ansv_hit<STRICT>(L.lv[k][j], v)) { found = true; break; }
        }
        if (found) {                       // descend: rightmost entry < v inside block j of level k
            while (k > 0) {
                uint64_t base = j * 32, end = base + 32;
                if (end > L.cnt[k - 1]) end = L.cnt[k - 1];
                uint64_t q = end;
                while (q > base) { q--; if (ansv_hit<STRICT>(L.lv[k - 1][q], v)) break; }
                j = q;
                k--;
            }
            return (uint32_t)j;
        }
        if (k + 1 >= L.nlev || (idx >> 5) == 0) {
            if (k + 1 >= L.nlev) return ANSV_NONE;
        }
        idx >>= 5;
        k++;
        if (k >= L.nlev) return ANSV_NONE;
        if (idx == 0) return ANSV_NONE;
    }
}
template <bool STRICT>
__device__ __forceinline__ uint64_t ansv_right(const AnsvLevels &L, uint64_t i, uint32_t v, uint64_t n) {
    uint64_t idx = i;
    int k = 0;
    while (true) {
        uint64_t last = (idx | 31) + 1;
        if (last > L.cnt[k]) last = L.cnt[k];
        uint64_t j = idx + 1;
        bool found = false;
        for (; j < last; j++) if (ansv_hit<STRICT>(L.lv[k][j], v)) { found = true; break; }
        if (found) {
            while (k > 0) {
                uint64_t base = j * 32, end = base + 32;
                if (end > L.cnt[k - 1]) end = L.cnt[k - 1];
                uint64_t q = base;
                while (q < end && !ansv_hit<STRICT>(L.lv[k - 1][q], v)) q++;
                j = q;
                k--;
            }
            return j;
        }
        idx >>= 5;
        k++;
        if (k >= L.nlev) return n;
    }
}
// STRICT = false gives the previous / next smaller-or-equal values; a null nsv skips the right side.
template <bool STRICT>
__global__ void __launch_bounds__(BLK) k_ansv(AnsvLevels L, uint64_t n, uint32_t *psv, uint32_t *nsv) {
    uint64_t i = (uint64_t)blockIdx.x * BLK + threadIdx.x;
    if (i >= n) return;
    uint32_t v = L.lv[0][i];
    psv[i] = ansv_left<STRICT>(L, i, v);
    if (nsv) nsv[i] = (uint32_t)ansv_right<STRICT>(L, i, v, n);
}

}  // namespace b200sa

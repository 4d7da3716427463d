// b200sa.cu -- context, level driver and C-ABI of libb200sa.so (sm_100a).
//
// Host-side level driver for the device pipeline that replaces
// `sais_table` / `sais` (reference src/table.rs:378-574) and
// `lcp_lens_quadratic` (src/table.rs:348-361).  See DESIGN.md for the phase
// map.  No CPU fallback exists: every entry point launches CUDA kernels or
// fails with an error code.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <string>
#include <vector>

#include "../../include/b200sa.h"
#include "../../include/b200sa_internal.h"
#include "common.cuh"
#include "classify.cuh"
#include "classify2.cuh"
#include "induce.cuh"
#include "induce2.cuh"
#include "induce3.cuh"
#include "induce4.cuh"
#include "induce5.cuh"
#include "induce6.cuh"
#include "pipeline_kernels.cuh"
#include "lms_sort.cuh"
#include "shard.cuh"
#include "tree.cuh"
#include "nccl_dyn.h"

using namespace b200sa;

// ---------------------------------------------------------------- context
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
};

struct b200sa_ctx {
    int device = 0;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;   // stream of the current call
    cudaStream_t copy_stream = nullptr;   // D2H of the SA overlapped with the LCP kernels
    cudaEvent_t ev_sa = nullptr;
    int sm_count = 0;
    int induce_blocks = 0;          // largest co-resident grid (workspace is sized for it)
    int induce_bps_max = 1;         // occupancy bound over all variants, blocks per SM
    int induce_occ[3] = {1, 1, 1};  // occupancy bound per text packing (2, 4, 8 bits) of the default variant
    int induce_occ_v[7][3] = {{1, 1, 1}, {1, 1, 1}, {1, 1, 1}, {1, 1, 1}, {1, 1, 1}, {1, 1, 1}, {1, 1, 1}};   // per kernel variant
    int induce_bps_env = 0;         // B200SA_INDUCE_BPS override (0 = adaptive)
    int cur_induce_blocks = 0;      // grid of the current build
    std::string last_error;
    bool timing = false;
    std::vector<std::pair<const char *, cudaEvent_t>> marks;
    std::vector<cudaEvent_t> event_pool;
    size_t events_used = 0;
    std::vector<const char *> phase_names;
    std::vector<float> phase_ms;
    b200sa_stats stats;
    uint32_t launches = 0;
    uint32_t *h_pin = nullptr;       // pinned read-back area (64 words)
    uint32_t *h_tab = nullptr;       // pinned copy of bstart[257] | Lcnt[256] (early SA copy-out)
    uint32_t *early_sa_out = nullptr;   // host SA buffer of the current host-API call (or null)
    bool early_done = false;
    size_t ws_bytes = 0;
    // ---- workspace
    DevBuf text, sa, lcp;                      // staging for the host API
    DevBuf pred, stype, lmsb, lmsrank, lmspos, lmslist, lmspred, sorted, flag, reduced, sa_r;
    DevBuf blkstate, carry, tables, small, scan_partial, radix_cnt, blkcnt;
    DevBuf os_hist, os_status, phik, phiv, runscr, plcp_samp;
    DevBuf k32b, k64a, k64b, v0, v1, p0, p1, g0, g1, rank, isa, qbuf;
    DevBuf packed, scan_state, cls_state, lmsdesc, steplog, hist_copies;
    uint32_t cls_calls = 0;
    // multi-GPU (SURVEY 8e): communicator owned or attached, NCCL resolved at run time
    ncclComm_t comm = nullptr;
    bool comm_owned = false;
    int nranks = 1, comm_rank = 0;
    DevBuf sh_a, sh_b, sh_c, sh_d, sh_e, sh_f, sh_small;
    DevBuf tree;                      // staging of the host suffix-tree API (six node arrays)
    bool lms_asc_ready = false;       // c->lmspos / c->lmsrank (text order) valid for the current text
    uint32_t scan_epoch = 0, scan_tiles_cap = 0;
    bool l2_persist = false;          // access policy window for the packed text (B200SA_L2PERSIST)
    size_t l2_max_window = 0, l2_set_aside = 0;
    uint32_t sigma = 256;            // distinct bytes of the current text
    int bits = 8;                    // bits per char of the packed text of the current call (2, 4 or 8 = raw)
    const void *ptext = nullptr;     // packed words, or the byte text when bits == 8
    uint64_t last_n = 0, last_m = 0;
};

// layout of the `tables` buffer (u32 words)
constexpr int T_BSTART = 0, T_LCNT = 257, T_SCNT = 513, T_LMSOFF = 769, T_HIST = 1026, T_CODE = 1794,
              T_ALPHA = 2050, T_END = 2306;

static const char *kVersion = "b200sa 0.1 (sm_100a)";

#define CU_TRY(ctx, expr)                                                                   \
    do {                                                                                    \
        cudaError_t e__ = (expr);                                                           \
        if (e__ != cudaSuccess) {                                                           \
            char buf__[512];                                                                \
            snprintf(buf__, sizeof buf__, "%s:%d: %s -> %s", __FILE__, __LINE__, #expr,     \
                     cudaGetErrorString(e__));                                              \
            (ctx)->last_error = buf__;                                                      \
            return (e__ == cudaErrorMemoryAllocation) ? B200SA_ERR_OOM : B200SA_ERR_CUDA;   \
        }                                                                                   \
    } while (0)

#define TRY(expr)                        \
    do {                                 \
        int rc__ = (expr);               \
        if (rc__ != B200SA_OK) return rc__; \
    } while (0)

static int ensure(b200sa_ctx *c, DevBuf &b, size_t bytes) {
    if (bytes == 0) bytes = 16;
    if (b.cap >= bytes) return B200SA_OK;
    if (b.p) { CU_TRY(c, cudaFree(b.p)); c->ws_bytes -= b.cap; b.p = nullptr; b.cap = 0; }
    size_t want = bytes + bytes / 16 + 256;    // a little slack against regrowth
    want = (want + 255) & ~(size_t)255;
    CU_TRY(c, cudaMalloc(&b.p, want));
    b.cap = want;
    c->ws_bytes += want;
    return B200SA_OK;
}
template <class T>
static T *ptr(DevBuf &b) { return reinterpret_cast<T *>(b.p); }

static inline uint32_t cdiv(uint64_t a, uint64_t b) { return (uint32_t)((a + b - 1) / b); }

static int mark(b200sa_ctx *c, const char *name) {
    if (!c->timing) return B200SA_OK;
    if (c->events_used == c->event_pool.size()) {
        cudaEvent_t e;
        CU_TRY(c, cudaEventCreate(&e));
        c->event_pool.push_back(e);
    }
    cudaEvent_t e = c->event_pool[c->events_used++];
    CU_TRY(c, cudaEventRecord(e, c->stream));
    c->marks.push_back({name, e});
    return B200SA_OK;
}
static void begin_call(b200sa_ctx *c, void *stream) {
    c->stream = stream ? (cudaStream_t)stream : c->own_stream;
    c->marks.clear();
    c->events_used = 0;
    c->launches = 0;
    c->last_error.clear();
}
static void l2_window(b200sa_ctx *c, const void *p, size_t bytes);
static int end_call(b200sa_ctx *c) {
    if (c->l2_persist) l2_window(c, nullptr, 0);              // the caller's stream leaves without our policy
    c->stats.kernel_launches = c->launches;
    c->stats.workspace_bytes = c->ws_bytes;
    c->phase_names.clear();
    c->phase_ms.clear();
    if (c->timing && c->marks.size() >= 2) {
        CU_TRY(c, cudaEventSynchronize(c->marks.back().second));
        for (size_t i = 0; i + 1 < c->marks.size(); i++) {
            float ms = 0;
            CU_TRY(c, cudaEventElapsedTime(&ms, c->marks[i].second, c->marks[i + 1].second));
            c->phase_names.push_back(c->marks[i].first);
            c->phase_ms.push_back(ms);
        }
    }
    return B200SA_OK;
}

template <class... KArgs, class... Args>
static inline void launch_k(b200sa_ctx *c, void (*kern)(KArgs...), uint32_t grid, Args... args) {
    kern<<<grid, BLK, 0, c->stream>>>(args...);
    c->launches++;
}
#define LAUNCH(ctx, kern, grid, ...) launch_k((ctx), kern, (grid), __VA_ARGS__)

static int read_words(b200sa_ctx *c, const uint32_t *dsrc, int count) {
    CU_TRY(c, cudaMemcpyAsync(c->h_pin, dsrc, sizeof(uint32_t) * count, cudaMemcpyDeviceToHost, c->stream));
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    return B200SA_OK;
}

// ------------------------------------------------------- generic primitives
// Single-pass scan (k_scan_lb, common.cuh): one launch, the input functor is evaluated once
// per element.  The tile descriptors live in c->scan_state and are epoch-tagged, so nothing
// is cleared between scans; a (re)allocated buffer is zeroed once (epochs start at 2).
// Scan descriptors for a kernel that embeds tile_lookback (same buffer and epochs as dev_scan).
static int scan_state_for(b200sa_ctx *c, uint32_t nb, ScanState *S) {
    size_t need = (size_t)nb * 28 + 64;
    if (c->scan_state.cap < need) {
        TRY(ensure(c, c->scan_state, need * 2));
        CU_TRY(c, cudaMemsetAsync(c->scan_state.p, 0, c->scan_state.cap, c->stream));
        c->scan_tiles_cap = (uint32_t)((c->scan_state.cap - 64) / 28);
    }
    uint8_t *basep = ptr<uint8_t>(c->scan_state);
    S->ticket = reinterpret_cast<uint32_t *>(basep);
    S->agg = reinterpret_cast<unsigned long long *>(basep + 64);
    S->incl = S->agg + c->scan_tiles_cap;
    S->pk = S->incl + c->scan_tiles_cap;
    S->flag = reinterpret_cast<uint32_t *>(S->pk + c->scan_tiles_cap);
    c->scan_epoch += 2;
    S->epoch = c->scan_epoch;
    return B200SA_OK;
}

template <class Op, class InF, class OutF>
static int dev_scan(b200sa_ctx *c, InF in, OutF out, uint64_t n, typename Op::T *d_total) {
    typedef typename Op::T T;
    if (n == 0) {
        if (d_total) CU_TRY(c, cudaMemsetAsync(d_total, 0, sizeof(T), c->stream));
        return B200SA_OK;
    }
    uint32_t nb = cdiv(n, SCAN_CHUNK);
    ScanState S;
    TRY(scan_state_for(c, nb, &S));
    LAUNCH(c, (k_scan_lb<Op, InF, OutF>), nb, in, out, n, nb, S, d_total);
    CU_TRY(c, cudaGetLastError());
    return B200SA_OK;
}

constexpr uint32_t MAX_RADIX_BLOCKS = 1184;   // 148 SMs x 8

template <class DigF, class MoveF>
static int radix_pass(b200sa_ctx *c, DigF dig, MoveF mv, uint64_t n) {
    if (n == 0) return B200SA_OK;
    uint32_t tiles = cdiv(n, TILE);
    uint32_t nb = tiles < MAX_RADIX_BLOCKS ? tiles : MAX_RADIX_BLOCKS;
    uint32_t tpb = cdiv(tiles, nb);
    nb = cdiv(tiles, tpb);
    TRY(ensure(c, c->radix_cnt, (size_t)256 * nb * 4));
    uint32_t *cnt = ptr<uint32_t>(c->radix_cnt);
    LAUNCH(c, (k_radix_hist<DigF>), nb, dig, n, tpb, cnt);
    TRY((dev_scan<OpSum>(c, InArray{cnt}, OutStoreExcl{cnt}, (uint64_t)256 * nb, nullptr)));
    LAUNCH(c, (k_radix_scatter<DigF, MoveF>), nb, dig, mv, n, tpb, cnt);
    CU_TRY(c, cudaGetLastError());
    return B200SA_OK;
}

// Sorts (ka,va) by the low `bits` of the key with the one-sweep passes of
// common.cuh; *kout/*vout point at the buffer pair holding the result.
template <class K, int OSI>
static int sort_pairs_t(b200sa_ctx *c, K *ka, uint32_t *va, K *kb, uint32_t *vb, uint64_t n, int bits,
                      K **kout, uint32_t **vout) {
    *kout = ka;
    *vout = va;
    if (n == 0 || bits <= 0) return B200SA_OK;
    int npass = (bits + 7) / 8;
    if (npass > OS_MAX_PASSES) npass = OS_MAX_PASSES;
    uint32_t tiles = cdiv(n, OSI * BLK);
    size_t status_bytes = (size_t)tiles * 256 * 8;
    TRY(ensure(c, c->os_hist, OS_MAX_PASSES * 256 * 4 + 64));
    TRY(ensure(c, c->os_status, status_bytes));
    uint32_t *ghist = ptr<uint32_t>(c->os_hist);
    uint32_t *ticket = ghist + OS_MAX_PASSES * 256;
    CU_TRY(c, cudaMemsetAsync(ghist, 0, OS_MAX_PASSES * 256 * 4 + 64, c->stream));
    uint32_t hb = cdiv(n, TILE) < 1184u ? cdiv(n, TILE) : 1184u;
    {
        size_t shm = (size_t)NWARP * npass * 256 * 4;
        auto kfn = k_os_hist<K, LoadArr<K>>;
        CU_TRY(c, cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(NWARP * OS_MAX_PASSES * 256 * 4)));
        kfn<<<hb, BLK, shm, c->stream>>>(LoadArr<K>{ka}, n, npass, 0u, ghist, (K *)nullptr);
        c->launches++;
    }
    LAUNCH(c, k_os_scan, (uint32_t)npass, ghist);
    for (int p = 0; p < npass; p++) {
        CU_TRY(c, cudaMemsetAsync(c->os_status.p, 0, status_bytes, c->stream));
        LAUNCH(c, (k_os_pass<K, LoadArr<K>, LoadArr<uint32_t>, OSI>), tiles, LoadArr<K>{ka}, LoadArr<uint32_t>{va}, kb, vb, n,
               (uint32_t)(8 * p), ghist + p * 256,
               reinterpret_cast<volatile unsigned long long *>(c->os_status.p), ticket + p);
        K *tk = ka; ka = kb; kb = tk;
        uint32_t *tv = va; va = vb; vb = tv;
    }
    CU_TRY(c, cudaGetLastError());
    *kout = ka;
    *vout = va;
    return B200SA_OK;
}

// Large inputs take wider tiles (16 keys per thread for 32-bit keys, 12 for 64-bit keys: what fits 48 KB of
// static shared memory): half the tiles, look-backs and per-tile scans per key (LMS sort 1.57 -> 1.44 ms).
template <class K>
static int sort_pairs(b200sa_ctx *c, K *ka, uint32_t *va, K *kb, uint32_t *vb, uint64_t n, int bits,
                      K **kout, uint32_t **vout) {
    if (n >= (1u << 20) && !getenv("B200SA_SORT_NARROW"))
        return sort_pairs_t<K, (sizeof(K) == 4 ? 16 : 12)>(c, ka, va, kb, vb, n, bits, kout, vout);
    return sort_pairs_t<K, ITEMS>(c, ka, va, kb, vb, n, bits, kout, vout);
}

// Same sort, but the first pass reads its (key, value) items from functors (no materialised
// input arrays); at least one pass runs, so the result always lands in a buffer pair.
template <class K, class KeyF, class ValF, int OSI = ITEMS>
static int sort_pairs_from(b200sa_ctx *c, KeyF keyf, ValF valf, K *ka, uint32_t *va, K *kb, uint32_t *vb, uint64_t n,
                           int bits, K **kout, uint32_t **vout) {
    *kout = ka;
    *vout = va;
    if (n == 0) return B200SA_OK;
    int npass = (bits + 7) / 8;
    if (npass < 1) npass = 1;
    if (npass > OS_MAX_PASSES) npass = OS_MAX_PASSES;
    uint32_t tiles = cdiv(n, OSI * BLK);
    size_t status_bytes = (size_t)tiles * 256 * 8;
    TRY(ensure(c, c->os_hist, OS_MAX_PASSES * 256 * 4 + 64));
    TRY(ensure(c, c->os_status, status_bytes));
    uint32_t *ghist = ptr<uint32_t>(c->os_hist);
    uint32_t *ticket = ghist + OS_MAX_PASSES * 256;
    CU_TRY(c, cudaMemsetAsync(ghist, 0, OS_MAX_PASSES * 256 * 4 + 64, c->stream));
    uint32_t hb = cdiv(n, TILE) < 1184u ? cdiv(n, TILE) : 1184u;
    {
        size_t shm = (size_t)NWARP * npass * 256 * 4;
        auto kfn = k_os_hist<K, KeyF>;
        CU_TRY(c, cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(NWARP * OS_MAX_PASSES * 256 * 4)));
        kfn<<<hb, BLK, shm, c->stream>>>(keyf, n, npass, 0u, ghist, kb);      // kb <- the keys (free until pass 2 writes it)
        c->launches++;
    }
    LAUNCH(c, k_os_scan, (uint32_t)npass, ghist);
    volatile unsigned long long *status = reinterpret_cast<volatile unsigned long long *>(c->os_status.p);
    CU_TRY(c, cudaMemsetAsync(c->os_status.p, 0, status_bytes, c->stream));
    LAUNCH(c, (k_os_pass<K, LoadArr<K>, ValF, OSI>), tiles, LoadArr<K>{kb}, valf, ka, va, n, 0u, ghist, status, ticket);
    for (int p = 1; p < npass; p++) {
        CU_TRY(c, cudaMemsetAsync(c->os_status.p, 0, status_bytes, c->stream));
        LAUNCH(c, (k_os_pass<K, LoadArr<K>, LoadArr<uint32_t>, OSI>), tiles, LoadArr<K>{ka}, LoadArr<uint32_t>{va}, kb, vb, n,
               (uint32_t)(8 * p), ghist + p * 256, status, ticket + p);
        K *tk = ka; ka = kb; kb = tk;
        uint32_t *tv = va; va = vb; vb = tv;
    }
    CU_TRY(c, cudaGetLastError());
    *kout = ka;
    *vout = va;
    return B200SA_OK;
}

static int bit_length(uint64_t x) {
    int b = 0;
    while (x) { b++; x >>= 1; }
    return b;
}

// ------------------------------------------------------- reduced problem
// Refinement rounds shared by both entry paths.  On entry the na active
// suffixes (members of non-singleton groups) are listed in asuf with their SA
// slots in c->p0 and group starts in c->g0; rank[] and sa_r hold the order by
// the first h symbols.
static int doubling_rounds(b200sa_ctx *c, uint32_t m, uint32_t na, uint32_t *asuf, uint32_t *ascratch, uint64_t h,
                           uint32_t *rounds_io, const uint32_t *names_arr = nullptr, uint32_t kgram = 0,
                           uint32_t bw = 0) {
    uint32_t *sa_r = ptr<uint32_t>(c->sa_r), *rank = ptr<uint32_t>(c->rank);
    uint32_t *apos = ptr<uint32_t>(c->p0), *apos_next = ptr<uint32_t>(c->p1);
    uint32_t *G0 = ptr<uint32_t>(c->g0), *G1 = ptr<uint32_t>(c->g1), *agrp = G0;
    uint32_t *d_na = ptr<uint32_t>(c->small);
    uint32_t rounds = *rounds_io;
    if (na > 0) {
        TRY(ensure(c, c->k64a, (size_t)na * 8));
        TRY(ensure(c, c->k64b, (size_t)na * 8));
    }
    int b2 = bit_length(m);
    bool try_local = getenv("B200SA_NO_LOCAL_SORT") == nullptr;
    static const char *kSortNames[] = {"rsa_sort1", "rsa_sort2", "rsa_sort3", "rsa_sort4", "rsa_sort5", "rsa_sortN"};
    static const char *kScanNames[] = {"rsa_scan1", "rsa_scan2", "rsa_scan3", "rsa_scan4", "rsa_scan5", "rsa_scanN"};
    while (na > 0) {
        rounds++;
        { uint32_t ri = rounds - *rounds_io; TRY(mark(c, kSortNames[ri <= 5 ? ri - 1 : 5])); }
        if (rounds > 40) { c->last_error = "doubling did not converge"; return B200SA_ERR_INTERNAL; }
        uint64_t *KA = ptr<uint64_t>(c->k64a), *KB = ptr<uint64_t>(c->k64b), *K2;
        uint32_t hh = h > 0xffffffffull ? 0xffffffffu : (uint32_t)h;
        bool first = (names_arr != nullptr) && rounds == *rounds_io + 1 && kgram >= 2;
        int bits = 2 * b2;
        if (first) {     // depth 1 -> depth kgram in one sort of kgram dense names
            LAUNCH(c, (k_multi_key_list<uint64_t>), cdiv(na, BLK), names_arr, m, asuf, na, kgram, bw, KA);
            bits = (int)(kgram * bw);
        } else {
            LAUNCH(c, k_pair_keys, cdiv(na, BLK), agrp, asuf, rank, na, m, hh, (uint32_t)b2, KA);
        }
        uint32_t *Vsorted = nullptr;
        bool sorted_locally = false;
        bool use_local = !first && try_local;
        if (use_local) {                        // probe ~4096 elements: are large groups common?
            CU_TRY(c, cudaMemsetAsync(d_na + 24, 0, 16, c->stream));   // [24] overflow, [25] large count, [26] max size
            uint32_t stride = na / 4096u; if (stride < 1) stride = 1;
            uint32_t samples = cdiv(na, stride);
            LAUNCH(c, k_group_probe, cdiv(samples, BLK), KA, na, (uint32_t)b2, stride, d_na + 25);
            TRY(read_words(c, d_na + 25, 2));
            if (c->h_pin[0] * 20u > samples) use_local = false;   // > 5 % of the elements in big groups: this round only
        }
        if (use_local) {                        // tiny groups: rank inside the group by counting
            LAUNCH(c, k_group_local_sort, cdiv(na, BLK), KA, asuf, na, (uint32_t)b2, KB, ascratch, d_na + 24);
            TRY(read_words(c, d_na + 24, 1));
            if (c->h_pin[0] == 0) { K2 = KB; Vsorted = ascratch; sorted_locally = true; }
            else try_local = false;             // some group is large: radix sort from now on
        }
        if (!sorted_locally) TRY(sort_pairs<uint64_t>(c, KA, asuf, KB, ascratch, na, bits, &K2, &Vsorted));
        uint32_t *Vother = (Vsorted == asuf) ? ascratch : asuf;
        { uint32_t ri = rounds - *rounds_io; TRY(mark(c, kScanNames[ri <= 5 ? ri - 1 : 5])); }
        TRY((dev_scan<OpMaxSum>(c, InGroupActive<uint64_t>{K2, apos, na},
                                OutGroupRankCompact{Vsorted, apos, rank, sa_r, apos_next, Vother, G0}, na,
                                reinterpret_cast<unsigned long long *>(d_na + 16))));
        TRY(read_words(c, d_na + 16, 1));          // low word of the pair total = number of ambiguous suffixes
        na = c->h_pin[0];
        if (getenv("B200SA_TRACE")) fprintf(stderr, "[b200sa] doubling round %u: h=%llu -> active %u of %u\n", rounds, (unsigned long long)h, na, m);
        asuf = Vother; ascratch = Vsorted;
        uint32_t *t = apos; apos = apos_next; apos_next = t;
        agrp = G0;
        if (first) h = kgram; else h *= 2;
    }
    *rounds_io = rounds;
    return B200SA_OK;
}


// SA of the u32 string R[0..m) (all symbols < names) -> ctx->sa_r.
// Stands in for the reference's recursion (src/table.rs:494-500): sort by
// name, then refine (group, rank[i+h]) pairs, doubling h, keeping only
// suffixes whose group is not yet a singleton.
static int reduced_sa(b200sa_ctx *c, uint32_t *R, uint32_t m, uint32_t names, uint32_t *rounds_out) {
    TRY(ensure(c, c->sa_r, (size_t)m * 4));
    TRY(ensure(c, c->k32b, (size_t)m * 4));
    TRY(ensure(c, c->v0, (size_t)m * 4));
    TRY(ensure(c, c->v1, (size_t)m * 4));
    TRY(ensure(c, c->p0, (size_t)m * 4));
    TRY(ensure(c, c->p1, (size_t)m * 4));
    TRY(ensure(c, c->g0, (size_t)m * 4));
    TRY(ensure(c, c->g1, (size_t)m * 4));
    TRY(ensure(c, c->rank, (size_t)m * 4));
    TRY(ensure(c, c->small, 256));
    uint32_t *sa_r = ptr<uint32_t>(c->sa_r), *rank = ptr<uint32_t>(c->rank);
    uint32_t *V0 = ptr<uint32_t>(c->v0), *V1 = ptr<uint32_t>(c->v1);
    uint32_t *P0 = ptr<uint32_t>(c->p0), *P1 = ptr<uint32_t>(c->p1);
    uint32_t *G0 = ptr<uint32_t>(c->g0), *G1 = ptr<uint32_t>(c->g1);
    uint32_t *d_na = ptr<uint32_t>(c->small);
    uint32_t rounds = 0;

    // round 0: sort suffixes by their first k symbols (k chosen so that the
    // key has about bit_length(m)+2 bits: random-like inputs become almost all
    // singletons after one sort; k = 1 when the alphabet is already ~m).
    LAUNCH(c, k_iota, cdiv(m, BLK), V0, m);
    int bm = bit_length(m);
    int bw = bit_length(names);               // symbols are stored +1 (0 = past the end)
    if (bw < 1) bw = 1;
    uint32_t k0 = 1;
    if (bw + 3 < bm) {
        k0 = (uint32_t)((bm + 2 + bw - 1) / bw);
        if ((int)k0 * bw > 64) k0 = 64 / bw;
    }
    if (const char *e = getenv("B200SA_K0")) { int v = atoi(e); if (v >= 1 && v * bw <= 64) k0 = (uint32_t)v; }
    uint32_t *Vs;
    uint32_t na = 0;
    if ((int)k0 * bw <= 32) {
        uint32_t *KA = ptr<uint32_t>(c->k32b), *Ks;
        LAUNCH(c, (k_multi_key<uint32_t>), cdiv(m, BLK), R, m, k0, (uint32_t)bw, KA);
        // R itself is the ping-pong partner (it is dead once the keys exist)
        TRY(sort_pairs<uint32_t>(c, KA, V0, R, V1, m, (int)k0 * bw, &Ks, &Vs));
        TRY((dev_scan<OpMax>(c, InGroupStart<uint32_t>{Ks, nullptr}, OutGroupRank{Vs, nullptr, G1, rank, sa_r}, m, nullptr)));
        uint32_t *Vf = (Vs == V0) ? V1 : V0;
        TRY((dev_scan<OpSum>(c, InActive<uint32_t>{Ks, m}, OutCompactActive{nullptr, Vs, G1, P0, Vf, G0}, m, d_na)));
    } else {
        TRY(ensure(c, c->k64a, (size_t)m * 8));
        TRY(ensure(c, c->k64b, (size_t)m * 8));
        uint64_t *KA = ptr<uint64_t>(c->k64a), *KB = ptr<uint64_t>(c->k64b), *Ks;
        LAUNCH(c, (k_multi_key<uint64_t>), cdiv(m, BLK), R, m, k0, (uint32_t)bw, KA);
        TRY(sort_pairs<uint64_t>(c, KA, V0, KB, V1, m, (int)k0 * bw, &Ks, &Vs));
        TRY((dev_scan<OpMax>(c, InGroupStart<uint64_t>{Ks, nullptr}, OutGroupRank{Vs, nullptr, G1, rank, sa_r}, m, nullptr)));
        uint32_t *Vf = (Vs == V0) ? V1 : V0;
        TRY((dev_scan<OpSum>(c, InActive<uint64_t>{Ks, m}, OutCompactActive{nullptr, Vs, G1, P0, Vf, G0}, m, d_na)));
    }
    uint32_t *Vfree = (Vs == V0) ? V1 : V0;
    TRY(read_words(c, d_na, 1));
    na = c->h_pin[0];
    TRY(doubling_rounds(c, m, na, Vfree, Vs, k0, &rounds));
    if (rounds_out) *rounds_out = rounds;
    return B200SA_OK;
}

// ------------------------------------------------------- L2 residency of the packed text
// The induce, the window keys of the LMS sort and the direct LCP all gather from the packed
// text at random while hundreds of MB of suffix-array data stream through L2.  An access
// policy window marks the packed text persisting (evict-last) for the kernels of this call.
static void l2_window(b200sa_ctx *c, const void *p, size_t bytes) {
    if (!c->l2_persist || c->l2_max_window == 0) return;
    cudaStreamAttrValue v;
    memset(&v, 0, sizeof v);
    v.accessPolicyWindow.base_ptr = const_cast<void *>(p);
    v.accessPolicyWindow.num_bytes = bytes < c->l2_max_window ? bytes : c->l2_max_window;
    v.accessPolicyWindow.hitRatio = bytes ? 1.0f : 0.0f;
    v.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
    v.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
    if (cudaStreamSetAttribute(c->stream, cudaStreamAttributeAccessPolicyWindow, &v) != cudaSuccess) cudaGetLastError();
}

// ------------------------------------------------------- packed text
// Chooses 2 / 4 bits per char when the alphabet allows it and packs the text;
// code_of/alpha live in the tables buffer.
static int pack_text(b200sa_ctx *c, const uint8_t *text, uint64_t n, uint32_t sigma) {
    uint32_t *tab = ptr<uint32_t>(c->tables);
    c->bits = 8;
    c->ptext = text;
    c->sigma = sigma;
    if (getenv("B200SA_NOPACK")) return B200SA_OK;
    if (sigma <= 4) c->bits = 2; else if (sigma <= 16) c->bits = 4; else return B200SA_OK;
    uint32_t cpw = 32 / c->bits;
    uint64_t words = (n + cpw - 1) / cpw;
    TRY(ensure(c, c->packed, words * 4 + 32));  // + padding for text_bits() / text_bits_wide()
    if (c->bits == 2) LAUNCH(c, (k_pack<2>), cdiv(words, BLK), text, n, tab + T_CODE, ptr<uint32_t>(c->packed));
    else LAUNCH(c, (k_pack<4>), cdiv(words, BLK), text, n, tab + T_CODE, ptr<uint32_t>(c->packed));
    CU_TRY(c, cudaGetLastError());
    c->ptext = c->packed.p;
    if (words * 4 <= c->l2_set_aside) l2_window(c, c->packed.p, words * 4 + 8);
    return B200SA_OK;
}

// ------------------------------------------------------- direct LMS-suffix sort
// lms_sort.cuh: radix sort of the LMS suffixes by character windows + refinement of the
// tied groups.  On success *list_out points at the LMS suffixes in suffix order (the
// seed of the final induce).  *done = false: the text has long repeats (groups stay tied);
// the caller takes the robust path (stage-1 induce, naming, rank doubling).
static uint32_t window_chars(uint32_t sigma, int bits, uint64_t *range_out) {
    if (bits == 2) { *range_out = 1ull << 32; return 16; }
    if (sigma < 2) sigma = 2;
    uint32_t cap = bits == 4 ? 13u : 8u, k = 0;
    uint64_t r = 1;
    while (k < cap && r * sigma <= (1ull << 32)) { r *= sigma; k++; }
    *range_out = r;
    return k;
}

template <int BITS>
static int lms_direct_sort_t(b200sa_ctx *c, uint32_t n, uint32_t m, uint32_t **list_out, bool *done) {
    *done = false;
    uint64_t range = 0;
    LmsWin W;
    W.ptext = c->ptext; W.code_of = ptr<uint32_t>(c->tables) + T_CODE; W.n = n;
    W.sigma = BITS == 2 ? 4u : c->sigma;
    W.kc = window_chars(c->sigma, BITS, &range);
    const uint32_t kc = W.kc;
    TRY(ensure(c, c->k32b, (size_t)m * 4));
    TRY(ensure(c, c->reduced, (size_t)m * 4));
    TRY(ensure(c, c->v0, (size_t)m * 4));
    TRY(ensure(c, c->v1, (size_t)m * 4));
    TRY(ensure(c, c->small, 4096));
    uint32_t *sm = ptr<uint32_t>(c->small);
    uint32_t *Ks, *Ps;
    TRY(mark(c, "lms_sort"));
    {
        const char *e = getenv("B200SA_SORT_ITEMS");            // keys per thread of the one-sweep passes: 8 | 16
        const bool wide = e ? atoi(e) == 16 : (m >= (1u << 20) && !getenv("B200SA_SORT_NARROW"));
        LmsKeyDesc<BITS> kf{W, ptr<uint32_t>(c->lmsdesc)};
        LmsValDesc vf{ptr<uint32_t>(c->lmsdesc)};
        if (wide)
            TRY((sort_pairs_from<uint32_t, LmsKeyDesc<BITS>, LmsValDesc, 16>(c, kf, vf, ptr<uint32_t>(c->k32b), ptr<uint32_t>(c->v0),
                                                                             ptr<uint32_t>(c->reduced), ptr<uint32_t>(c->v1), m,
                                                                             bit_length(range - 1), &Ks, &Ps)));
        else
            TRY((sort_pairs_from<uint32_t, LmsKeyDesc<BITS>, LmsValDesc, ITEMS>(c, kf, vf, ptr<uint32_t>(c->k32b), ptr<uint32_t>(c->v0),
                                                                                ptr<uint32_t>(c->reduced), ptr<uint32_t>(c->v1), m,
                                                                                bit_length(range - 1), &Ks, &Ps)));
    }
    // groups of equal windows; members of non-singleton groups -> active list
    TRY(mark(c, "lms_groups"));
    TRY(ensure(c, c->p0, (size_t)m * 4));
    TRY(ensure(c, c->p1, (size_t)m * 4));
    TRY(ensure(c, c->g0, (size_t)m * 4));
    TRY(ensure(c, c->g1, (size_t)m * 4));
    TRY(ensure(c, c->sa_r, (size_t)m * 4));
    TRY(ensure(c, c->rank, (size_t)m * 4));
    uint32_t *slotA = ptr<uint32_t>(c->p0), *slotB = ptr<uint32_t>(c->p1);
    uint32_t *grpA = ptr<uint32_t>(c->g0), *grpB = ptr<uint32_t>(c->g1);
    uint32_t *posA = ptr<uint32_t>(c->sa_r), *posB = ptr<uint32_t>(c->rank);
    unsigned long long *d_tot = reinterpret_cast<unsigned long long *>(sm + 16);
    {
        size_t fw = ((size_t)m + 31) / 32 + 1;
        TRY(ensure(c, c->flag, fw * 4));
        uint32_t *forced = ptr<uint32_t>(c->flag);
        CU_TRY(c, cudaMemsetAsync(forced, 0, fw * 4, c->stream));
        CU_TRY(c, cudaMemsetAsync(sm + 16, 0, 8, c->stream));
        LAUNCH(c, (k_lms_mark_trunc<BITS>), 1u, W, ptr<uint32_t>(c->lmsdesc), m, Ks, Ps, kc, forced);
        if (getenv("B200SA_GROUPS_GENERIC")) {       // the generic scan with functors (cross-check)
            InLmsActive1 in1{Ks, forced, m};
            TRY((dev_scan<OpSum>(c, in1, OutLmsCompact1{in1, Ps, slotA, posA, grpA}, m, sm + 16)));
        } else {
            uint32_t nt = cdiv(m, LG_TILE);
            ScanState S;
            TRY(scan_state_for(c, nt, &S));
            LAUNCH(c, k_lms_groups1, nt, Ks, Ps, forced, m, nt, S, slotA, posA, grpA, sm + 16);
            CU_TRY(c, cudaGetLastError());
        }
    }
    TRY(read_words(c, sm + 16, 1));
    uint32_t na = c->h_pin[0];
    c->stats.names = m - na;                       // LMS suffixes settled by the first window
    uint32_t rounds = 1;
    uint32_t max_rounds = BITS == 8 ? 16u : 8u;    // byte windows hold 4-8 chars: natural text needs ~10 of them
    if (const char *e = getenv("B200SA_DIRECT_ROUNDS")) { int v = atoi(e); if (v >= 1) max_rounds = (uint32_t)v; }
    if (getenv("B200SA_TRACE")) fprintf(stderr, "[b200sa] direct LMS sort: kc=%u, round 1 leaves %u of %u tied\n", kc, na, m);
    const bool force = getenv("B200SA_DIRECT_FORCE") != nullptr;            // experiments: never bail out early
    // the window tells (almost) nothing apart: every suffix has a twin for kc characters -- repeats, not
    // a skewed alphabet (English leaves 99.5 % tied after 5 bytes and still converges in ~10 rounds)
    if (!force && (uint64_t)na * 1000 > (uint64_t)m * 999 && m > 64) return B200SA_OK;
    if (na > 0)     // group id of every tied element = slot of its group's head
        TRY((dev_scan<OpMax>(c, InArray{grpA}, OutMaxInPlace{grpA}, na, nullptr)));
    uint64_t h = kc;
    const bool allow_local = getenv("B200SA_NO_LOCAL_SORT") == nullptr;
    const int gbits = 32 + bit_length(m);
    while (na > 0) {
        if (rounds >= max_rounds) return B200SA_OK;            // still tied: robust path
        rounds++;
        {
            static const char *kNames[] = {"lms_refine2", "lms_refine3", "lms_refine4", "lms_refine5", "lms_refineN"};
            TRY(mark(c, kNames[rounds - 2 < 4 ? rounds - 2 : 4]));
        }
        TRY(ensure(c, c->k64a, (size_t)na * 8));
        TRY(ensure(c, c->k64b, (size_t)na * 8));
        TRY(ensure(c, c->sorted, (size_t)m * 4));
        uint64_t *KA = ptr<uint64_t>(c->k64a), *KB = ptr<uint64_t>(c->k64b), *K2 = nullptr;
        uint32_t *scratch = ptr<uint32_t>(c->sorted), *P2 = nullptr;
        LAUNCH(c, (k_lms_refine_keys<BITS>), cdiv(na, BLK), W, posA, grpA, na, (uint32_t)h, KA);
        const uint32_t span = (uint32_t)(h + kc > 0xffffffffull ? 0xffffffffull : h + kc);
        bool local_ok = false;
        bool try_local = allow_local;
        if (try_local && na >= (1u << 20)) {    // probe ~4096 elements: counting inside a group is quadratic in its size
                                                // (a short list is cheap either way: no probe, no extra host round trip)
            CU_TRY(c, cudaMemsetAsync(sm + 24, 0, 16, c->stream));   // [24] overflow, [25] members of big groups, [26] max size
            uint32_t stride = na / 4096u; if (stride < 1) stride = 1;
            uint32_t samples = cdiv(na, stride);
            LAUNCH(c, k_group_probe, cdiv(samples, BLK), KA, na, 32u, stride, sm + 25);
            TRY(read_words(c, sm + 25, 2));
            if (c->h_pin[0] * 20u > samples) try_local = false;     // > 5 % of the elements sit in groups of >= 128
        }
        if (try_local) {                         // tiny groups: rank inside the group by counting
            CU_TRY(c, cudaMemsetAsync(sm + 24, 0, 4, c->stream));
            LAUNCH(c, k_group_local_sort, cdiv(na, BLK), KA, posA, na, 32u, KB, scratch, sm + 24);
            TRY((dev_scan<OpMaxSum>(c, InLmsGroupR{KB, scratch, slotA, na, n, span},
                                    OutLmsCompactR{scratch, slotA, Ps, slotB, posB, grpB}, na, d_tot)));
            TRY(read_words(c, sm + 16, 9));          // [0] tied count ... [8] = sm[24] overflow flag
            local_ok = c->h_pin[8] == 0;             // some group larger than the limit: radix sort this round
        }
        if (!local_ok) {
            TRY(sort_pairs<uint64_t>(c, KA, posA, KB, scratch, na, gbits, &K2, &P2));
            // (posA may now hold sorted values; the compaction below writes posB)
            TRY((dev_scan<OpMaxSum>(c, InLmsGroupR{K2, P2, slotA, na, n, span},
                                    OutLmsCompactR{P2, slotA, Ps, slotB, posB, grpB}, na, d_tot)));
            TRY(read_words(c, sm + 16, 1));
        }
        uint32_t na_next = c->h_pin[0];
        if (getenv("B200SA_TRACE")) fprintf(stderr, "[b200sa] direct LMS sort: round %u (h=%llu): %u -> %u tied\n", rounds, (unsigned long long)h, na, na_next);
        // slow convergence on a large residue means long repeats: stop early
        if (!force && (uint64_t)na_next * 100 > (uint64_t)na * 85 && (uint64_t)na_next * 64 > m) return B200SA_OK;
        na = na_next;
        uint32_t *t;
        t = slotA; slotA = slotB; slotB = t;
        t = posA; posA = posB; posB = t;
        t = grpA; grpA = grpB; grpB = t;
        h += kc;
    }
    c->stats.doubling_rounds = rounds;
    *list_out = Ps;
    *done = true;
    return B200SA_OK;
}
static int lms_direct_sort(b200sa_ctx *c, uint32_t n, uint32_t m, uint32_t **list_out, bool *done) {
    if (c->bits == 2) return lms_direct_sort_t<2>(c, n, m, list_out, done);
    if (c->bits == 4) return lms_direct_sort_t<4>(c, n, m, list_out, done);
    return lms_direct_sort_t<8>(c, n, m, list_out, done);
}

// ------------------------------------------------------- induce launcher
// Kernel variants of the induce passes (profiles/README.md compares them; B200SA_INDUCE=1..6 forces one):
//   1  one-round steps with MATCH ranking (any packing; the default for 4-bit and byte text)
//   2  multi-round bucket steps (packed text)
//   3  packed-counter ranking on physically aligned tiles (2-bit text)
//   4  3 + three carried predecessor chars per byte + staged coalesced stores (2-bit text)
//   5  warp-private tile streams + 16-bit carried chars with producer-side refresh (2-bit text)
//   6  3's block-wide tiles + 5's carried chars + cascade steps for short chain lists (2-bit text; default there;
//      B200SA_NO_CASCADE / B200SA_CASCADE_MAX=<entries> switch the cascade steps off / limit them)
static int induce_variant_env() {
    const char *e = getenv("B200SA_INDUCE");       // read per call: tests switch variants inside one process
    return e ? atoi(e) : 0;
}
static int induce_variant(int bits) {
    int v = induce_variant_env();
    if (v == 2 && bits < 8) return 2;
    if (v == 1) return 1;
    if (bits == 2) return (v >= 3 && v <= 5) ? v : 6;
    return 1;
}
static const void *induce_fn_v(bool spass, int bits, int variant) {
    if (variant == 6 && bits == 2) return spass ? (const void *)k_induce6<true> : (const void *)k_induce6<false>;
    if (variant == 5 && bits == 2) return spass ? (const void *)k_induce5<true> : (const void *)k_induce5<false>;
    if (variant == 4 && bits == 2) return spass ? (const void *)k_induce4<true> : (const void *)k_induce4<false>;
    if (variant == 3 && bits == 2) return spass ? (const void *)k_induce3<true> : (const void *)k_induce3<false>;
    if (variant == 2 && bits == 2) return spass ? (const void *)k_induce2<true, 2> : (const void *)k_induce2<false, 2>;
    if (variant == 2 && bits == 4) return spass ? (const void *)k_induce2<true, 4> : (const void *)k_induce2<false, 4>;
    if (bits == 2) return spass ? (const void *)k_induce<true, 2> : (const void *)k_induce<false, 2>;
    if (bits == 4) return spass ? (const void *)k_induce<true, 4> : (const void *)k_induce<false, 4>;
    return spass ? (const void *)k_induce<true, 8> : (const void *)k_induce<false, 8>;
}
static int launch_induce(b200sa_ctx *c, bool spass, const uint8_t *text, uint32_t n, uint32_t *sa,
                         const uint32_t *lms, uint32_t m) {
    (void)m;
    uint32_t *tab = ptr<uint32_t>(c->tables);
    InduceArgs A;
    A.text = text; A.ptext = c->ptext; A.alpha = tab + T_ALPHA;
    A.n = n; A.sa = sa; A.pred = ptr<uint8_t>(c->pred);
    A.lms = lms; A.lms_pred = ptr<uint8_t>(c->lmspred);
    A.bstart = tab + T_BSTART; A.Lcnt = tab + T_LCNT; A.Scnt = tab + T_SCNT; A.lms_off = tab + T_LMSOFF;
    A.blk_cnt = ptr<uint32_t>(c->blkcnt);
    uint32_t *sm = ptr<uint32_t>(c->small);
    A.g_fill = sm + 64; A.g_state = reinterpret_cast<int32_t *>(sm + 320); A.err = sm + 32;
    A.run_scratch = ptr<uint32_t>(c->runscr);
    A.run_alive = A.run_scratch + TILE;
    A.cmd = sm + 336;
    A.steplog = nullptr;
    A.blocklog_step = 0;
    A.carry = 0;
    { static int rs = -1; if (rs < 0) { const char *e = getenv("B200SA_RUN_STREAK"); rs = e ? atoi(e) : 0; } A.run_streak = (uint32_t)rs; }
    if (getenv("B200SA_STEPLOG")) {
        if (ensure(c, c->steplog, 8192 * 8) == B200SA_OK) {
            A.steplog = ptr<unsigned long long>(c->steplog);
            if (const char *e = getenv("B200SA_BLOCKLOG")) {          // "<pass 0|1>:<big step index>"
                int ps = 0, st = 0;
                if (sscanf(e, "%d:%d", &ps, &st) == 2 && ps == (spass ? 1 : 0)) A.blocklog_step = (uint32_t)st + 1u;
            }
            if (!spass) cudaMemsetAsync(c->steplog.p, 0, 8, c->stream);
        }
    }
    void *args[] = {&A};
    int variant = induce_variant(c->bits);
    if (variant >= 3 && (((uintptr_t)sa | (uintptr_t)lms) & 15) != 0) variant = 1;      // 16-byte loads need aligned arrays
    A.carry = (variant >= 5) ? 2 : (variant == 4 ? 1 : 0);
    int bi = c->bits == 2 ? 0 : (c->bits == 4 ? 1 : 2);
    int blocks = c->cur_induce_blocks, cap = c->sm_count * c->induce_occ_v[variant][bi];
    if (blocks > cap) blocks = cap;
    A.cascade = 0;
    if (variant == 6 && !getenv("B200SA_NO_CASCADE")) {          // multi-round steps for the short lists of every bucket's cascade
        A.cascade = (uint32_t)blocks * (uint32_t)TILE;
        if (const char *e = getenv("B200SA_CASCADE_MAX")) { long v = atol(e); if (v >= 0 && (uint64_t)v < A.cascade) A.cascade = (uint32_t)v; }
    }
    CU_TRY(c, cudaLaunchCooperativeKernel(induce_fn_v(spass, c->bits, variant), dim3(blocks), dim3(BLK), args, 0, c->stream));
    c->launches++;
    return B200SA_OK;
}

// ------------------------------------------------------- the level driver
// After the histogram is known: packed text and the grid of the persistent induce kernels.
static int post_classify(b200sa_ctx *c, const uint8_t *text, uint64_t n, uint32_t sigma) {
    TRY(pack_text(c, text, n, sigma));
    // few buckets -> long lists, latency bound -> more blocks per SM; many buckets -> grid-sync bound -> one per SM
    int bps = sigma <= 16 ? 3 : (sigma <= 64 ? 2 : 1);
    if (c->induce_bps_env) bps = c->induce_bps_env;
    int occ_here = c->induce_occ[c->bits == 2 ? 0 : (c->bits == 4 ? 1 : 2)];
    if (bps > occ_here) bps = occ_here;
    if (bps < 1) bps = 1;
    c->cur_induce_blocks = c->sm_count * bps;
    return B200SA_OK;
}

// K1 fused (classify2.cuh): one pass -> type / LMS bitmaps, (byte, type) histogram, bucket
// tables, LMS positions in descending text order (c->lmsdesc), packed text.
static int classify_fused_dev(b200sa_ctx *c, const uint8_t *text, uint64_t n, uint32_t *m_out,
                              ShardEdge edge = ShardEdge{-1, -1, ST_L}, bool pack = true) {
    uint64_t nw = (n + 31) / 32;
    uint32_t nbc = cdiv(nw, CLS_WORDS);
    TRY(ensure(c, c->stype, nw * 4));
    TRY(ensure(c, c->lmsb, nw * 4));
    TRY(ensure(c, c->tables, T_END * 4));
    TRY(ensure(c, c->small, 4096));
    TRY(ensure(c, c->lmsdesc, (size_t)(n / 2 + 2) * 4));
    if (c->cls_state.cap < (size_t)nbc * 4) {
        TRY(ensure(c, c->cls_state, (size_t)nbc * 8));
        CU_TRY(c, cudaMemsetAsync(c->cls_state.p, 0, c->cls_state.cap, c->stream));
    }
    uint32_t *tab = ptr<uint32_t>(c->tables), *hist = tab + T_HIST, *sm = ptr<uint32_t>(c->small);
    TRY(ensure(c, c->hist_copies, (size_t)HIST_COPIES * 768 * 4));
    CU_TRY(c, cudaMemsetAsync(c->hist_copies.p, 0, (size_t)HIST_COPIES * 768 * 4, c->stream));
    CU_TRY(c, cudaMemsetAsync(sm, 0, 4096, c->stream));
    ScanState S;
    TRY(scan_state_for(c, nbc, &S));
    Cls2State CS{ptr<uint32_t>(c->cls_state), (++c->cls_calls) * 8u};
    // B200SA_CLASSIFY_TMA=1: the tile arrives by one cp.async.bulk (UBLKCP) + mbarrier instead of 512 vector
    // loads.  Measured on 100 MB G_dna: 0.43 ms vs 0.42 ms -- with ~5 resident one-tile CTAs per SM the load
    // latency is already covered, so the bulk copy buys nothing here and stays opt-in.
    if (getenv("B200SA_CLASSIFY_TMA") == nullptr)
        LAUNCH(c, k_classify_fused<false>, nbc, text, n, nbc, S, CS, ptr<uint32_t>(c->stype), ptr<uint32_t>(c->lmsb),
               ptr<uint32_t>(c->hist_copies), ptr<uint32_t>(c->lmsdesc), sm, edge);
    else
        LAUNCH(c, k_classify_fused<true>, nbc, text, n, nbc, S, CS, ptr<uint32_t>(c->stype), ptr<uint32_t>(c->lmsb),
               ptr<uint32_t>(c->hist_copies), ptr<uint32_t>(c->lmsdesc), sm, edge);
    LAUNCH(c, k_hist_fold, 1u, ptr<uint32_t>(c->hist_copies), hist);
    LAUNCH(c, k_bucket_tables, 1, hist, tab + T_BSTART, tab + T_LCNT, tab + T_SCNT, tab + T_LMSOFF, tab + T_CODE,
           tab + T_ALPHA, sm + 3);
    CU_TRY(c, cudaGetLastError());
    if (c->early_sa_out)
        CU_TRY(c, cudaMemcpyAsync(c->h_tab, tab + T_BSTART, 513 * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
    TRY(read_words(c, sm, 4));
    uint32_t m = c->h_pin[0], sigma = c->h_pin[3];
    if (pack) TRY(post_classify(c, text, n, sigma));
    c->lms_asc_ready = false;
    *m_out = m;
    return B200SA_OK;
}

// Text-order LMS positions + per-word LMS ranks (robust path, k_unrename): derived on demand.
static int lms_ascending(b200sa_ctx *c, uint64_t n, uint32_t m) {
    if (c->lms_asc_ready) return B200SA_OK;
    uint64_t nw = (n + 31) / 32;
    TRY(ensure(c, c->lmsrank, nw * 4));
    TRY(ensure(c, c->lmspos, (size_t)m * 4));
    TRY((dev_scan<OpSum>(c, InPopcWords{ptr<uint32_t>(c->lmsb)}, OutStoreExcl{ptr<uint32_t>(c->lmsrank)}, nw, nullptr)));
    if (m > 0) LAUNCH(c, k_reverse_u32, cdiv(m, BLK), ptr<uint32_t>(c->lmsdesc), m, ptr<uint32_t>(c->lmspos));
    CU_TRY(c, cudaGetLastError());
    c->lms_asc_ready = true;
    return B200SA_OK;
}


static int classify_dev(b200sa_ctx *c, const uint8_t *text, uint64_t n, uint32_t *m_out,
                        ShardEdge edge = ShardEdge{-1, -1, ST_L}) {
    uint64_t nw = (n + 31) / 32;
    uint32_t nbc = cdiv(nw, CLS_WORDS);
    TRY(ensure(c, c->stype, nw * 4));
    TRY(ensure(c, c->lmsb, nw * 4));
    TRY(ensure(c, c->lmsrank, nw * 4));
    TRY(ensure(c, c->blkstate, nbc));
    TRY(ensure(c, c->carry, nbc));
    TRY(ensure(c, c->tables, T_END * 4));
    TRY(ensure(c, c->small, 4096));
    uint32_t *tab = ptr<uint32_t>(c->tables);
    uint32_t *hist = tab + T_HIST;
    uint32_t *sm = ptr<uint32_t>(c->small);
    CU_TRY(c, cudaMemsetAsync(hist, 0, 768 * 4, c->stream));
    CU_TRY(c, cudaMemsetAsync(sm, 0, 4096, c->stream));
    LAUNCH(c, k_cls_block_state, nbc, text, n, ptr<uint8_t>(c->blkstate), edge);
    LAUNCH(c, k_cls_carry, 1, ptr<uint8_t>(c->blkstate), nbc, ptr<uint8_t>(c->carry), edge.next_char >= 0 ? edge.tail_carry : ST_L);
    LAUNCH(c, k_cls_types, nbc, text, n, ptr<uint8_t>(c->carry), ptr<uint32_t>(c->stype), ptr<uint32_t>(c->lmsb), hist, edge);
    LAUNCH(c, k_bucket_tables, 1, hist, tab + T_BSTART, tab + T_LCNT, tab + T_SCNT, tab + T_LMSOFF, tab + T_CODE,
           tab + T_ALPHA, sm + 3);
    CU_TRY(c, cudaGetLastError());
    TRY((dev_scan<OpSum>(c, InPopcWords{ptr<uint32_t>(c->lmsb)}, OutStoreExcl{ptr<uint32_t>(c->lmsrank)}, nw, sm)));
    if (c->early_sa_out)    // bucket layout for the early SA copy-out (same synchronisation as the read below)
        CU_TRY(c, cudaMemcpyAsync(c->h_tab, tab + T_BSTART, 513 * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
    TRY(read_words(c, sm, 4));
    uint32_t m = c->h_pin[0], sigma = c->h_pin[3];
    TRY(post_classify(c, text, n, sigma));
    TRY(ensure(c, c->lmspos, (size_t)m * 4));
    if (m > 0) {
        LAUNCH(c, k_lms_positions, cdiv(nw, BLK), ptr<uint32_t>(c->lmsb), ptr<uint32_t>(c->lmsrank), nw, ptr<uint32_t>(c->lmspos));
        CU_TRY(c, cudaGetLastError());
    }
    c->lms_asc_ready = true;
    *m_out = m;
    return B200SA_OK;
}

// Host API only: the L parts of all buckets are final after the last L pass and the
// S parts after the last S pass, so the SA can start leaving over PCIe one S-pass
// early (few buckets only: one memcpy per bucket part).
static int early_copy_parts(b200sa_ctx *c, const uint32_t *d_sa, bool s_parts) {
    if (!c->early_sa_out || c->sigma > 16) return B200SA_OK;
    CU_TRY(c, cudaEventRecord(c->ev_sa, c->stream));
    CU_TRY(c, cudaStreamWaitEvent(c->copy_stream, c->ev_sa, 0));
    const uint32_t *bstart = c->h_tab, *Lcnt = c->h_tab + 257;
    for (int b = 0; b < 256; b++) {
        uint32_t lo = bstart[b] + (s_parts ? Lcnt[b] : 0u);
        uint32_t hi = s_parts ? bstart[b + 1] : bstart[b] + Lcnt[b];
        if (hi > lo)
            CU_TRY(c, cudaMemcpyAsync(c->early_sa_out + lo, d_sa + lo, (size_t)(hi - lo) * 4, cudaMemcpyDeviceToHost, c->copy_stream));
    }
    if (s_parts) c->early_done = true;
    return B200SA_OK;
}

static int build_dev(b200sa_ctx *c, const uint8_t *d_text, uint64_t n, uint32_t *d_sa) {
    memset(&c->stats, 0, sizeof c->stats);
    c->stats.n = n;
    c->stats.sm_count = c->sm_count;
    c->stats.induce_blocks = c->induce_blocks;   // updated after classification
    c->last_n = n; c->last_m = 0;
    if (n > B200SA_MAX_N) { c->last_error = "text longer than 2^32-4096 bytes"; return B200SA_ERR_TOO_LARGE; }
    if (n == 0) return B200SA_OK;
    if (n == 1) { CU_TRY(c, cudaMemsetAsync(d_sa, 0, 4, c->stream)); return B200SA_OK; }
    const uint8_t *text = d_text;
    if (((uintptr_t)d_text & 15) != 0) {       // vector loads need 16-byte alignment
        TRY(ensure(c, c->text, n));
        CU_TRY(c, cudaMemcpyAsync(c->text.p, d_text, n, cudaMemcpyDeviceToDevice, c->stream));
        text = ptr<uint8_t>(c->text);
    }
    uint32_t n32 = (uint32_t)n;
    TRY(mark(c, "classify"));
    uint32_t m = 0;
    if (getenv("B200SA_CLASSIFY_V1")) {          // three-kernel classifier (classify.cuh) + reversed position list
        TRY(classify_dev(c, text, n, &m));
        TRY(ensure(c, c->lmsdesc, (size_t)m * 4 + 16));
        if (m > 0) LAUNCH(c, k_reverse_u32, cdiv(m, BLK), ptr<uint32_t>(c->lmspos), m, ptr<uint32_t>(c->lmsdesc));
    } else {
        TRY(classify_fused_dev(c, text, n, &m));
    }
    c->stats.m = m; c->last_m = m;
    c->stats.induce_blocks = c->cur_induce_blocks;
    TRY(ensure(c, c->pred, 2 * n + 64));          // bytes (variants 1-4) or 16-bit carried words (variant 5)
    TRY(ensure(c, c->lmslist, (size_t)m * 4));
    TRY(ensure(c, c->lmspred, 2 * (size_t)m + 64));
    TRY(ensure(c, c->blkcnt, (size_t)2 * c->induce_blocks * 256 * 4));
    TRY(ensure(c, c->runscr, (size_t)2 * TILE * 4));
    uint32_t *lmslist = ptr<uint32_t>(c->lmslist);
    bool direct_done = false;
    if (m > 0 && !getenv("B200SA_NO_DIRECT")) {
        uint32_t *lst = nullptr;
        TRY(lms_direct_sort(c, n32, m, &lst, &direct_done));
        if (direct_done) lmslist = lst;
    }
    c->stats.direct_sort = direct_done ? 1u : 0u;
    if (m > 0 && !direct_done) {
        c->stats.doubling_rounds = 0;
        TRY(lms_ascending(c, n, m));              // text-order positions + per-word ranks for the robust path
        TRY(ensure(c, c->sorted, (size_t)m * 4));
        TRY(ensure(c, c->flag, m));
        TRY(ensure(c, c->reduced, (size_t)m * 4));
        uint32_t *sm = ptr<uint32_t>(c->small);
        // K3: LMS suffixes grouped by first byte (stable, text order inside a group)
        TRY(mark(c, "lms_group"));
        TRY(radix_pass(c, DigTextAtPos{text, ptr<uint32_t>(c->lmspos)}, MoveU32{ptr<uint32_t>(c->lmspos), lmslist}, m));
        // stage 1: induced sort of the LMS substrings
        TRY(mark(c, "induce1_L"));
        TRY(launch_induce(c, false, text, n32, d_sa, lmslist, m));
        TRY(mark(c, "induce1_S"));
        TRY(launch_induce(c, true, text, n32, d_sa, lmslist, m));
        // K6: sorted LMS substrings
        TRY(mark(c, "compact_lms"));
        TRY((dev_scan<OpSum>(c, InIsLmsEntry{d_sa, ptr<uint32_t>(c->lmsb)}, OutCompactSa{d_sa, ptr<uint32_t>(c->sorted)}, n, sm + 1)));
        // K7/K8: names, reduced string
        TRY(mark(c, "name"));
        if (c->bits == 2)
            LAUNCH(c, (k_name_flags<2>), cdiv(m, BLK), c->ptext, n32, ptr<uint32_t>(c->lmsb),
                   ptr<uint32_t>(c->sorted), m, ptr<uint8_t>(c->flag));
        else if (c->bits == 4)
            LAUNCH(c, (k_name_flags<4>), cdiv(m, BLK), c->ptext, n32, ptr<uint32_t>(c->lmsb),
                   ptr<uint32_t>(c->sorted), m, ptr<uint8_t>(c->flag));
        else
            LAUNCH(c, (k_name_flags<8>), cdiv(m, BLK), c->ptext, n32, ptr<uint32_t>(c->lmsb),
                   ptr<uint32_t>(c->sorted), m, ptr<uint8_t>(c->flag));
        TRY((dev_scan<OpSum>(c, InFlagU8{ptr<uint8_t>(c->flag)},
                             OutReduced{ptr<uint32_t>(c->sorted), ptr<uint32_t>(c->lmsb), ptr<uint32_t>(c->lmsrank), ptr<uint32_t>(c->reduced)},
                             m, sm + 2)));
        TRY(read_words(c, sm + 1, 2));
        uint32_t cnt_lms = c->h_pin[0], names = c->h_pin[1];
        if (cnt_lms != m) {
            char b[160]; snprintf(b, sizeof b, "stage-1 induce lost LMS entries: %u of %u", cnt_lms, m);
            c->last_error = b; return B200SA_ERR_INTERNAL;
        }
        c->stats.names = names;
        // K8/K9 + recursion stand-in: the sorted LMS substrings already give the
        // reduced suffixes ordered by their first symbol, so doubling starts at
        // h = 1 without sorting the names again.
        TRY(mark(c, "reduced_sa"));
        TRY(ensure(c, c->sa_r, (size_t)m * 4));
        TRY(ensure(c, c->rank, (size_t)m * 4));
        TRY(ensure(c, c->g1, (size_t)m * 4));
        // first refinement: k-gram of dense names (reduced string), k = as many as fit 64 bits
        uint32_t bw = (uint32_t)bit_length(names);
        uint32_t kgram = bw ? 64u / bw : 0u;
        if (kgram > 8) kgram = 8;
        if (const char *e = getenv("B200SA_KGRAM")) { int v = atoi(e); if (v >= 0 && (uint32_t)v * bw <= 64) kgram = (uint32_t)v; }
        TRY((dev_scan<OpMax>(c, InFlagPos{ptr<uint8_t>(c->flag)},
                             OutInitFromSorted{ptr<uint32_t>(c->sorted), ptr<uint32_t>(c->lmsb), ptr<uint32_t>(c->lmsrank),
                                               ptr<uint8_t>(c->flag), m, kgram >= 2 ? 0 : 1,
                                               ptr<uint32_t>(c->sa_r), ptr<uint32_t>(c->g1), ptr<uint32_t>(c->rank)},
                             m, nullptr)));
        if (names < m) {
            TRY(ensure(c, c->v0, (size_t)m * 4));
            TRY(ensure(c, c->v1, (size_t)m * 4));
            TRY(ensure(c, c->p0, (size_t)m * 4));
            TRY(ensure(c, c->p1, (size_t)m * 4));
            TRY(ensure(c, c->g0, (size_t)m * 4));
            TRY((dev_scan<OpSum>(c, InActive<uint32_t>{ptr<uint32_t>(c->g1), m},
                                 OutCompactActive{nullptr, ptr<uint32_t>(c->sa_r), ptr<uint32_t>(c->g1),
                                                  ptr<uint32_t>(c->p0), ptr<uint32_t>(c->v0), ptr<uint32_t>(c->g0)},
                                 m, sm)));
            TRY(read_words(c, sm, 1));
            uint32_t na = c->h_pin[0], rounds = 0;
            TRY(doubling_rounds(c, m, na, ptr<uint32_t>(c->v0), ptr<uint32_t>(c->v1), 1, &rounds,
                                ptr<uint32_t>(c->reduced), kgram, bw));
            c->stats.doubling_rounds = rounds;
        }
        // K10: ranks -> text positions; the list is grouped by first byte by construction
        TRY(mark(c, "unrename"));
        LAUNCH(c, k_unrename, cdiv(m, BLK), ptr<uint32_t>(c->sa_r), ptr<uint32_t>(c->lmspos), m, lmslist);
        CU_TRY(c, cudaGetLastError());
    }
    // stage 2: final induce from the sorted LMS suffixes
    TRY(mark(c, "induce2_L"));
    TRY(launch_induce(c, false, text, n32, d_sa, lmslist, m));
    TRY(early_copy_parts(c, d_sa, false));
    TRY(mark(c, "induce2_S"));
    TRY(launch_induce(c, true, text, n32, d_sa, lmslist, m));
    TRY(early_copy_parts(c, d_sa, true));
    TRY(mark(c, "end"));
    TRY(read_words(c, ptr<uint32_t>(c->small) + 32, 4));
    if (c->h_pin[0] != 0) {
        char b[200];
        snprintf(b, sizeof b, "induce invariant violated: bucket %u filled %u, expected %u", c->h_pin[1], c->h_pin[2], c->h_pin[3]);
        c->last_error = b;
        return B200SA_ERR_INTERNAL;
    }
    return B200SA_OK;
}

// k_lcp_direct on the packed text of the current call; pairs that reach `cap` (and could go on)
// are counted in *capped.  cap >= n computes every pair in full.
static void lcp_direct_launch(b200sa_ctx *c, uint32_t n32, const uint32_t *d_sa, uint32_t *d_lcp, uint32_t cap,
                              uint32_t *capped) {
    int lk = 2;       // runs of 32 ranks per warp = window gathers in flight per lane (2-bit text: 1 / 2 / 4 ->
                      // 0.66 / 0.57 / 0.59 ms per 10^8 ranks; 4-bit text is best with 1)
    if (const char *e = getenv("B200SA_LCP_K")) lk = atoi(e);
    if (c->bits == 2 && lk == 4) LAUNCH(c, (k_lcp_direct<2, 4>), cdiv(n32, BLK * 4), c->ptext, n32, d_sa, d_lcp, cap, capped);
    else if (c->bits == 2 && lk == 2) LAUNCH(c, (k_lcp_direct<2, 2>), cdiv(n32, BLK * 2), c->ptext, n32, d_sa, d_lcp, cap, capped);
    else if (c->bits == 2) LAUNCH(c, (k_lcp_direct<2, 1>), cdiv(n32, BLK), c->ptext, n32, d_sa, d_lcp, cap, capped);
    else if (c->bits == 4) LAUNCH(c, (k_lcp_direct<4, 1>), cdiv(n32, BLK), c->ptext, n32, d_sa, d_lcp, cap, capped);
    else LAUNCH(c, (k_lcp_direct<8, 1>), cdiv(n32, BLK), c->ptext, n32, d_sa, d_lcp, cap, capped);
}

// Is a caller table that passed the permutation check THE suffix array of the n bytes at d_text?
// inv (n u32) is scratch.  One scatter, one pass over the ranks, one word read back.
static int sa_is_sorted(b200sa_ctx *c, const uint8_t *d_text, uint64_t n, const uint32_t *d_sa, uint32_t *inv,
                        bool *sorted) {
    uint32_t n32 = (uint32_t)n;
    TRY(ensure(c, c->small, 4096));
    uint32_t *bad = ptr<uint32_t>(c->small) + 14;
    CU_TRY(c, cudaMemsetAsync(bad, 0, 4, c->stream));
    LAUNCH(c, k_sa_inverse, cdiv(n, BLK), d_sa, n32, inv);
    LAUNCH(c, k_sa_sorted, cdiv(n, BLK), d_text, n32, d_sa, inv, bad);
    TRY(read_words(c, bad, 1));
    *sorted = c->h_pin[0] == 0;
    return B200SA_OK;
}

// reuse_pack: the table was built by this call (fused build_lcp*) and the packed text is ready.
// Otherwise the table comes from the caller: it is checked to be a permutation, and before the
// Phi / PLCP path (only valid on the sorted table) to be the suffix array; a permutation that is
// not gets lcp_lens_quadratic's per-pair compare, uncapped.  require_sorted: reject a table that is
// not the suffix array (B200SA_ERR_BAD_ARG) instead.
static int lcp_dev(b200sa_ctx *c, const uint8_t *d_text, uint64_t n, const uint32_t *d_sa, uint32_t *d_lcp,
                   bool reuse_pack, bool require_sorted = false) {
    if (n > B200SA_MAX_N) return B200SA_ERR_TOO_LARGE;
    if (n == 0) return B200SA_OK;
    uint32_t n32 = (uint32_t)n;
    TRY(ensure(c, c->isa, (size_t)n * 4));
    if (!reuse_pack) {
        // stand-alone call: the table comes from the caller (from_parts accepts anything,
        // src/table.rs:111-119, and the reference would merely panic on a bad index), and
        // every LCP kernel indexes text and phi with sa[r]: check that it is a permutation
        // of 0..n-1 before trusting it
        TRY(mark(c, "lcp_validate"));
        TRY(ensure(c, c->small, 4096));
        uint64_t nwv = (n + 31) / 32;
        uint32_t *seen = ptr<uint32_t>(c->isa);             // free until the Phi path needs it
        uint32_t *bad = ptr<uint32_t>(c->small) + 12;
        CU_TRY(c, cudaMemsetAsync(seen, 0, nwv * 4, c->stream));
        CU_TRY(c, cudaMemsetAsync(bad, 0, 4, c->stream));
        CU_TRY(c, cudaMemsetAsync(bad + 1, 0, 4, c->stream));
        LAUNCH(c, k_sa_validate, cdiv(cdiv(n, 4), BLK), d_sa, n32, seen, bad);
        LAUNCH(c, k_sa_validate_count, 592u, seen, n32, bad + 1);
        LAUNCH(c, k_sa_validate_verdict, 1u, bad + 1, n32, bad);
        TRY(read_words(c, bad, 1));
        if (c->h_pin[0] != 0) {
            c->last_error = "table is not a permutation of 0..n-1 (index out of range or repeated)";
            return B200SA_ERR_BAD_ARG;
        }
    }
    if (!reuse_pack) {
        // stand-alone call: byte histogram -> alphabet -> packed text
        TRY(mark(c, "lcp_pack"));
        const uint8_t *text = d_text;
        if (((uintptr_t)d_text & 15) != 0) {
            TRY(ensure(c, c->text, n));
            CU_TRY(c, cudaMemcpyAsync(c->text.p, d_text, n, cudaMemcpyDeviceToDevice, c->stream));
            text = ptr<uint8_t>(c->text);
        }
        TRY(ensure(c, c->tables, T_END * 4));
        TRY(ensure(c, c->small, 4096));
        uint32_t *tab = ptr<uint32_t>(c->tables), *sm = ptr<uint32_t>(c->small);
        CU_TRY(c, cudaMemsetAsync(tab + T_HIST, 0, 256 * 4, c->stream));
        uint32_t hb = cdiv(n, BLK * 64);
        if (hb > 1184) hb = 1184;
        LAUNCH(c, k_byte_hist, hb, text, n, tab + T_HIST);
        LAUNCH(c, k_alpha_from_hist, 1, tab + T_HIST, tab + T_CODE, tab + T_ALPHA, sm + 3);
        TRY(read_words(c, sm + 3, 1));
        TRY(pack_text(c, text, n, c->h_pin[0]));
    }
    bool checked = false;
    if (require_sorted) {
        TRY(mark(c, "lcp_sorted"));
        bool sorted = false;
        TRY(sa_is_sorted(c, d_text, n, d_sa, ptr<uint32_t>(c->isa), &sorted));
        if (!sorted) {
            c->last_error = "table is not the suffix array of the text (adjacent suffixes out of order)";
            return B200SA_ERR_BAD_ARG;
        }
        checked = true;
    }
    // fast path: direct adjacent-pair compare when the text is L2-resident
    // (packed, or small); falls through to the linear path if any pair hits the cap
    if ((c->bits < 8 || n <= (32u << 20)) && !getenv("B200SA_LCP_LINEAR")) {
        TRY(mark(c, "lcp_direct"));
        TRY(ensure(c, c->small, 4096));
        uint32_t *sm = ptr<uint32_t>(c->small);
        CU_TRY(c, cudaMemsetAsync(sm + 8, 0, 4, c->stream));
        lcp_direct_launch(c, n32, d_sa, d_lcp, 256u, sm + 8);
        TRY(read_words(c, sm + 8, 1));
        if (c->h_pin[0] == 0) {
            TRY(mark(c, "end"));
            CU_TRY(c, cudaGetLastError());
            return B200SA_OK;
        }
    }
    if (!reuse_pack && !checked) {
        // a caller table about to take the linear path: Kasai's carry is only valid on the
        // suffix array; any other permutation gets the reference's quadratic per-pair compare
        TRY(mark(c, "lcp_sorted"));
        bool sorted = false;
        TRY(sa_is_sorted(c, d_text, n, d_sa, ptr<uint32_t>(c->isa), &sorted));
        if (!sorted) {
            TRY(mark(c, "lcp_unsorted"));
            lcp_direct_launch(c, n32, d_sa, d_lcp, n32, ptr<uint32_t>(c->small) + 8);
            TRY(mark(c, "end"));
            CU_TRY(c, cudaGetLastError());
            return B200SA_OK;
        }
    }
    TRY(mark(c, "lcp_phi"));
    if (n >= (1u << 22) && !getenv("B200SA_PHI_DIRECT")) {
        // partition (sa[r], sa[r-1]) by the top byte of sa[r], then scatter window by window
        TRY(ensure(c, c->phik, (size_t)n * 4));
        TRY(ensure(c, c->phiv, (size_t)n * 4));
        TRY(ensure(c, c->os_hist, OS_MAX_PASSES * 256 * 4 + 64));
        uint32_t tiles = cdiv(n, TILE);
        size_t status_bytes = (size_t)tiles * 256 * 8;
        TRY(ensure(c, c->os_status, status_bytes));
        uint32_t *ghist = ptr<uint32_t>(c->os_hist), *ticket = ghist + OS_MAX_PASSES * 256;
        int nbits = bit_length(n - 1);
        uint32_t shift = nbits > 8 ? (uint32_t)(nbits - 8) : 0u;
        CU_TRY(c, cudaMemsetAsync(ghist, 0, OS_MAX_PASSES * 256 * 4 + 64, c->stream));
        CU_TRY(c, cudaMemsetAsync(c->os_status.p, 0, status_bytes, c->stream));
        // sa is a permutation: the digit bases are known without a histogram pass
        LAUNCH(c, k_os_perm_base, 1u, ghist, shift, n32);
        LAUNCH(c, (k_os_pass<uint32_t, LoadArr<uint32_t>, LoadPhiPrev>), tiles, LoadArr<uint32_t>{d_sa}, LoadPhiPrev{d_sa},
               ptr<uint32_t>(c->phik), ptr<uint32_t>(c->phiv), n, shift, ghist,
               reinterpret_cast<volatile unsigned long long *>(c->os_status.p), ticket);
        LAUNCH(c, k_phi_apply, cdiv(n, BLK), ptr<uint32_t>(c->phik), ptr<uint32_t>(c->phiv), n32, ptr<uint32_t>(c->isa));
    } else {
        LAUNCH(c, k_phi, cdiv(n, BLK), d_sa, n32, ptr<uint32_t>(c->isa));
    }
    TRY(mark(c, "lcp_plcp"));
    uint32_t nchunk = cdiv(n, LCP_CHUNK);
    uint32_t pg = cdiv(nchunk, BLK), sg = cdiv(cdiv(nchunk, 32), BLK);
    TRY(ensure(c, c->plcp_samp, (size_t)nchunk * 4));
    uint32_t *samp = ptr<uint32_t>(c->plcp_samp), *phi = ptr<uint32_t>(c->isa);
    if (c->bits == 2) LAUNCH(c, (k_plcp_samples<2>), sg, c->ptext, n32, phi, samp, (uint64_t)0, ~(uint64_t)0);
    else if (c->bits == 4) LAUNCH(c, (k_plcp_samples<4>), sg, c->ptext, n32, phi, samp, (uint64_t)0, ~(uint64_t)0);
    else LAUNCH(c, (k_plcp_samples<8>), sg, c->ptext, n32, phi, samp, (uint64_t)0, ~(uint64_t)0);
    TRY(mark(c, "lcp_plcp_fill"));
    if (c->bits == 2) LAUNCH(c, (k_plcp<2>), pg, c->ptext, n32, phi, samp, (uint64_t)0, ~(uint64_t)0);
    else if (c->bits == 4) LAUNCH(c, (k_plcp<4>), pg, c->ptext, n32, phi, samp, (uint64_t)0, ~(uint64_t)0);
    else LAUNCH(c, (k_plcp<8>), pg, c->ptext, n32, phi, samp, (uint64_t)0, ~(uint64_t)0);
    TRY(mark(c, "lcp_gather"));
    LAUNCH(c, k_lcp_gather, cdiv(n, BLK), d_sa, ptr<uint32_t>(c->isa), n32, d_lcp);
    TRY(mark(c, "end"));
    CU_TRY(c, cudaGetLastError());
    return B200SA_OK;
}

template <class K>
static int test_sort(b200sa_ctx *c, K *keys, uint32_t *vals, uint64_t n, int bits) {
    if (!c || (n > 0 && (!keys || !vals))) return B200SA_ERR_BAD_ARG;
    CU_TRY(c, cudaSetDevice(c->device));
    begin_call(c, nullptr);
    TRY(ensure(c, c->k64a, n * sizeof(K)));
    TRY(ensure(c, c->k64b, n * sizeof(K)));
    TRY(ensure(c, c->v0, n * 4));
    TRY(ensure(c, c->v1, n * 4));
    CU_TRY(c, cudaMemcpyAsync(c->k64a.p, keys, n * sizeof(K), cudaMemcpyHostToDevice, c->stream));
    CU_TRY(c, cudaMemcpyAsync(c->v0.p, vals, n * 4, cudaMemcpyHostToDevice, c->stream));
    K *ko; uint32_t *vo;
    TRY(sort_pairs<K>(c, ptr<K>(c->k64a), ptr<uint32_t>(c->v0), ptr<K>(c->k64b), ptr<uint32_t>(c->v1), n, bits, &ko, &vo));
    if (n) {
        CU_TRY(c, cudaMemcpyAsync(keys, ko, n * sizeof(K), cudaMemcpyDeviceToHost, c->stream));
        CU_TRY(c, cudaMemcpyAsync(vals, vo, n * 4, cudaMemcpyDeviceToHost, c->stream));
    }
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    return end_call(c);
}

// ================================================================= C ABI
extern "C" {

const char *b200sa_version(void) { return kVersion; }

const char *b200sa_strerror(int code) {
    switch (code) {
        case B200SA_OK: return "ok";
        case B200SA_ERR_BAD_ARG: return "bad argument";
        case B200SA_ERR_TOO_LARGE: return "text longer than B200SA_MAX_N = 2^32-4096 bytes";
        case B200SA_ERR_NO_DEVICE: return "no usable CUDA device";
        case B200SA_ERR_OOM: return "out of device memory";
        case B200SA_ERR_CUDA: return "CUDA error";
        case B200SA_ERR_INTERNAL: return "internal invariant violated";
        default: return "unknown error";
    }
}

const char *b200sa_last_error(b200sa_ctx *ctx) { return ctx ? ctx->last_error.c_str() : "null context"; }

int b200sa_ctx_create(int device, b200sa_ctx **out) {
    if (!out) return B200SA_ERR_BAD_ARG;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) return B200SA_ERR_NO_DEVICE;
    if (device < 0 || device >= count) return B200SA_ERR_BAD_ARG;
    if (cudaSetDevice(device) != cudaSuccess) return B200SA_ERR_NO_DEVICE;
    b200sa_ctx *c = new b200sa_ctx();
    c->device = device;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { delete c; return B200SA_ERR_CUDA; }
    c->sm_count = prop.multiProcessorCount;
    if (const char *e = getenv("B200SA_L2FETCH")) {   // experiment: L2 fetch granularity for random gathers
        int v = atoi(e);
        if (v == 32 || v == 64 || v == 128) cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, (size_t)v);
    }
    if (!prop.cooperativeLaunch) { delete c; return B200SA_ERR_NO_DEVICE; }
    if (const char *e = getenv("B200SA_L2PERSIST")) {
        int mb = atoi(e);                                       // MB of L2 set aside for persisting lines
        if (mb > 0 && prop.persistingL2CacheMaxSize > 0) {
            size_t want = (size_t)mb << 20;
            if (want > (size_t)prop.persistingL2CacheMaxSize) want = (size_t)prop.persistingL2CacheMaxSize;
            if (cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, want) == cudaSuccess) {
                c->l2_persist = true;
                c->l2_set_aside = want;
                c->l2_max_window = (size_t)prop.accessPolicyMaxWindowSize;
            } else cudaGetLastError();
        }
    }
    if (cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking) != cudaSuccess) { delete c; return B200SA_ERR_CUDA; }
    c->stream = c->own_stream;
    if (cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&c->ev_sa, cudaEventDisableTiming) != cudaSuccess) { delete c; return B200SA_ERR_CUDA; }
    if (cudaMallocHost((void **)&c->h_pin, 64 * sizeof(uint32_t)) != cudaSuccess) { delete c; return B200SA_ERR_CUDA; }
    if (cudaMallocHost((void **)&c->h_tab, 513 * sizeof(uint32_t)) != cudaSuccess) { cudaFreeHost(c->h_pin); delete c; return B200SA_ERR_CUDA; }
    int occ = 0;
    {
        const int bb[3] = {2, 4, 8};
        for (int v = 1; v <= 6; v++)
            for (int k = 0; k < 3; k++) {
                int ok = 1 << 30;
                for (int sp = 0; sp < 2; sp++) {
                    int o = 0;
                    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o, induce_fn_v(sp != 0, bb[k], v), BLK, 0);
                    if (o < ok) ok = o;
                }
                c->induce_occ_v[v][k] = ok > 4 ? 4 : ok;
            }
        for (int k = 0; k < 3; k++) {
            c->induce_occ[k] = c->induce_occ_v[induce_variant(bb[k])][k];
            for (int v = 1; v <= 6; v++) if (c->induce_occ_v[v][k] > occ) occ = c->induce_occ_v[v][k];
        }
    }
    if (occ < 1) { cudaFreeHost(c->h_pin); delete c; return B200SA_ERR_CUDA; }
    c->induce_bps_max = occ > 4 ? 4 : occ;
    if (const char *e = getenv("B200SA_INDUCE_BPS")) { int v = atoi(e); if (v >= 1) c->induce_bps_env = v > occ ? occ : v; }
    c->induce_blocks = c->sm_count * c->induce_bps_max;
    c->cur_induce_blocks = c->sm_count;
    memset(&c->stats, 0, sizeof c->stats);
    *out = c;
    return B200SA_OK;
}

void b200sa_ctx_destroy(b200sa_ctx *c) {
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->comm && c->comm_owned && nccl_api().ok) nccl_api().CommDestroy(c->comm);
    DevBuf *bufs[] = {&c->text, &c->sa, &c->lcp, &c->pred, &c->stype, &c->lmsb, &c->lmsrank, &c->lmspos, &c->lmslist,
                      &c->lmspred, &c->sorted, &c->flag, &c->reduced, &c->sa_r, &c->blkstate, &c->carry, &c->tables,
                      &c->small, &c->scan_partial, &c->radix_cnt, &c->blkcnt, &c->k32b, &c->k64a, &c->k64b, &c->v0,
                      &c->v1, &c->p0, &c->p1, &c->g0, &c->g1, &c->rank, &c->isa, &c->qbuf, &c->os_hist, &c->os_status, &c->packed, &c->phik, &c->phiv, &c->runscr, &c->plcp_samp, &c->scan_state, &c->cls_state, &c->lmsdesc, &c->steplog, &c->hist_copies, &c->sh_a, &c->sh_b, &c->sh_c, &c->sh_d, &c->sh_e, &c->sh_f, &c->sh_small, &c->tree};
    for (DevBuf *b : bufs) if (b->p) cudaFree(b->p);
    for (cudaEvent_t e : c->event_pool) cudaEventDestroy(e);
    if (c->h_pin) cudaFreeHost(c->h_pin);
    if (c->h_tab) cudaFreeHost(c->h_tab);
    if (c->own_stream) cudaStreamDestroy(c->own_stream);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    if (c->ev_sa) cudaEventDestroy(c->ev_sa);
    delete c;
}

int b200sa_set_timing(b200sa_ctx *c, int enabled) {
    if (!c) return B200SA_ERR_BAD_ARG;
    c->timing = enabled != 0;
    return B200SA_OK;
}

int b200sa_last_phase_times(b200sa_ctx *c, const char **names, float *ms, int cap) {
    if (!c) return B200SA_ERR_BAD_ARG;
    int k = (int)c->phase_names.size();
    for (int i = 0; i < k && i < cap; i++) {
        if (names) names[i] = c->phase_names[i];
        if (ms) ms[i] = c->phase_ms[i];
    }
    return k;
}

int b200sa_last_stats(b200sa_ctx *c, b200sa_stats *out) {
    if (!c || !out) return B200SA_ERR_BAD_ARG;
    *out = c->stats;
    out->workspace_bytes = c->ws_bytes;
    return B200SA_OK;
}

int b200sa_build_dev(b200sa_ctx *c, const uint8_t *d_text, uint64_t n, uint32_t *d_sa, void *stream) {
    if (!c || (n > 0 && (!d_text || !d_sa))) return B200SA_ERR_BAD_ARG;
    CU_TRY(c, cudaSetDevice(c->device));
    begin_call(c, stream);
    int rc = build_dev(c, d_text, n, d_sa);
    if (rc == B200SA_OK) rc = end_call(c);
    return rc;
}

int b200sa_lcp_dev(b200sa_ctx *c, const uint8_t *d_text, uint64_t n, const uint32_t *d_sa, uint32_t *d_lcp,
                   void *stream) {
    if (!c || (n > 0 && (!d_text || !d_sa || !d_lcp))) return B200SA_ERR_BAD_ARG;
    CU_TRY(c, cudaSetDevice(c->device));
    begin_call(c, stream);
    int rc = lcp_dev(c, d_text, n, d_sa, d_lcp, false);
    if (rc == B200SA_OK) rc = end_call(c);
    return rc;
}

int b200sa_build_lcp_dev(b200sa_ctx *c, const uint8_t *d_text, uint64_t n, uint32_t *d_sa, uint32_t *d_lcp,
                         void *stream) {
    if (!c || (n > 0 && (!d_text || !d_sa || !d_lcp))) return B200SA_ERR_BAD_ARG;
    CU_TRY(c, cudaSetDevice(c->device));
    begin_call(c, stream);
    int rc = build_dev(c, d_text, n, d_sa);
    if (rc == B200SA_OK) {
        // build_dev may have classified an aligned copy of the text; the packed text (or that
        // copy) is still valid, so the LCP kernels reuse it (n >= 2 means classification ran)
        const uint8_t *t = (((uintptr_t)d_text & 15) != 0 && n >= 2) ? ptr<uint8_t>(c->text) : d_text;
        b200sa_stats st = c->stats;
        rc = lcp_dev(c, t, n, d_sa, d_lcp, n >= 2);
        c->stats = st;
    }
    if (rc == B200SA_OK) rc = end_call(c);
    return rc;
}

static int host_build_inner(b200sa_ctx *c, const uint8_t *text, uint64_t n, uint32_t *sa_out, uint32_t *lcp_out,
                            const uint32_t *sa_in) {
    if (n > B200SA_MAX_N) { c->last_error = "text longer than 2^32-4096 bytes"; return B200SA_ERR_TOO_LARGE; }
    CU_TRY(c, cudaSetDevice(c->device));
    begin_call(c, nullptr);
    memset(&c->stats, 0, sizeof c->stats);
    c->stats.n = n;
    if (n == 0) return end_call(c);
    TRY(ensure(c, c->text, n));
    TRY(ensure(c, c->sa, (size_t)n * 4));
    TRY(mark(c, "h2d"));
    CU_TRY(c, cudaMemcpyAsync(c->text.p, text, n, cudaMemcpyHostToDevice, c->stream));
    if (sa_in) CU_TRY(c, cudaMemcpyAsync(c->sa.p, sa_in, (size_t)n * 4, cudaMemcpyHostToDevice, c->stream));
    if (!sa_in) {
        // early copy-out only into pinned memory: a D2H into pageable memory blocks the host
        // thread, which would delay the launch of the last S pass
        bool pinned = false;
        if (sa_out) {
            cudaPointerAttributes pa;
            if (cudaPointerGetAttributes(&pa, sa_out) == cudaSuccess) pinned = (pa.type == cudaMemoryTypeHost);
            else cudaGetLastError();
        }
        c->early_sa_out = (pinned && n >= 2 && !getenv("B200SA_NO_EARLY_COPY")) ? sa_out : nullptr;
        c->early_done = false;
        int brc = build_dev(c, ptr<uint8_t>(c->text), n, ptr<uint32_t>(c->sa));
        c->early_sa_out = nullptr;
        if (brc != B200SA_OK) return brc;
        if (sa_out && c->early_done) {
            TRY(mark(c, "d2h_sa"));      // already on its way on the copy stream
        } else if (sa_out) {
            TRY(mark(c, "d2h_sa"));
            if (lcp_out) {      // the LCP kernels only read the SA: copy it out underneath them
                CU_TRY(c, cudaEventRecord(c->ev_sa, c->stream));
                CU_TRY(c, cudaStreamWaitEvent(c->copy_stream, c->ev_sa, 0));
                CU_TRY(c, cudaMemcpyAsync(sa_out, c->sa.p, (size_t)n * 4, cudaMemcpyDeviceToHost, c->copy_stream));
            } else {
                CU_TRY(c, cudaMemcpyAsync(sa_out, c->sa.p, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
            }
        }
    }
    if (lcp_out) {
        TRY(ensure(c, c->lcp, (size_t)n * 4));
        TRY(lcp_dev(c, ptr<uint8_t>(c->text), n, ptr<uint32_t>(c->sa), ptr<uint32_t>(c->lcp), sa_in == nullptr && n >= 2));
        TRY(mark(c, "d2h_lcp"));
        CU_TRY(c, cudaMemcpyAsync(lcp_out, c->lcp.p, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
    }
    TRY(mark(c, "end"));
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    CU_TRY(c, cudaStreamSynchronize(c->copy_stream));
    return end_call(c);
}

// Every exit of the host API passes through here: on failure, D2H copies into the caller's
// buffers may still be in flight on either stream, and the caller is free to release the
// buffers as soon as we return.
static int host_build(b200sa_ctx *c, const uint8_t *text, uint64_t n, uint32_t *sa_out, uint32_t *lcp_out,
                      const uint32_t *sa_in) {
    int rc = host_build_inner(c, text, n, sa_out, lcp_out, sa_in);
    if (rc != B200SA_OK) {
        c->early_sa_out = nullptr;
        if (c->stream) cudaStreamSynchronize(c->stream);
        if (c->copy_stream) cudaStreamSynchronize(c->copy_stream);
        cudaGetLastError();
    }
    return rc;
}

int b200sa_build(b200sa_ctx *c, const uint8_t *text, uint64_t n, uint32_t *sa_out) {
    if (!c || (n > 0 && (!text || !sa_out))) return B200SA_ERR_BAD_ARG;
    return host_build(c, text, n, sa_out, nullptr, nullptr);
}

int b200sa_lcp(b200sa_ctx *c, const uint8_t *text, uint64_t n, const uint32_t *sa, uint32_t *lcp_out) {
    if (!c || (n > 0 && (!text || !sa || !lcp_out))) return B200SA_ERR_BAD_ARG;
    return host_build(c, text, n, nullptr, lcp_out, sa);
}

int b200sa_build_lcp(b200sa_ctx *c, const uint8_t *text, uint64_t n, uint32_t *sa_out, uint32_t *lcp_out) {
    if (!c || (n > 0 && (!text || !sa_out || !lcp_out))) return B200SA_ERR_BAD_ARG;
    return host_build(c, text, n, sa_out, lcp_out, nullptr);
}

int b200sa_positions_dev(b200sa_ctx *c, const uint8_t *d_text, uint64_t n, const uint32_t *d_sa,
                         const uint8_t *d_queries, const uint64_t *d_q_off, uint32_t nq, uint32_t *d_start,
                         uint32_t *d_end, void *stream) {
    if (!c || (nq > 0 && (!d_q_off || !d_start || !d_end)) || (n > 0 && (!d_text || !d_sa))) return B200SA_ERR_BAD_ARG;
    if (n > B200SA_MAX_N) return B200SA_ERR_TOO_LARGE;
    CU_TRY(c, cudaSetDevice(c->device));
    begin_call(c, stream);
    if (nq > 0) {
        LAUNCH(c, k_positions, cdiv(nq, BLK), d_text, (uint32_t)n, d_sa, d_queries, d_q_off, nq, d_start, d_end);
        CU_TRY(c, cudaGetLastError());
    }
    return end_call(c);
}

// ------------------------------------------------------------ multi-GPU shards (SURVEY 8e)
int b200sa_shard_summary(b200sa_ctx *c, const uint8_t *d_shard, uint64_t len, int next_char, int *state_out, void *stream) {
    if (!c || !d_shard || len < 1 || len > B200SA_MAX_N || !state_out || next_char > 255) return B200SA_ERR_BAD_ARG;
    if (((uintptr_t)d_shard & 15) != 0) { c->last_error = "shard pointer must be 16-byte aligned"; return B200SA_ERR_BAD_ARG; }
    CU_TRY(c, cudaSetDevice(c->device));
    begin_call(c, stream);
    uint64_t nw = (len + 31) / 32;
    uint32_t nbc = cdiv(nw, CLS_WORDS);
    TRY(ensure(c, c->blkstate, nbc));
    TRY(ensure(c, c->carry, nbc));
    TRY(ensure(c, c->small, 4096));
    ShardEdge edge{next_char, -1, ST_P};
    LAUNCH(c, k_cls_block_state, nbc, d_shard, len, ptr<uint8_t>(c->blkstate), edge);
    LAUNCH(c, k_cls_carry, 1, ptr<uint8_t>(c->blkstate), nbc, ptr<uint8_t>(c->carry), (uint32_t)ST_P);
    CU_TRY(c, cudaGetLastError());
    uint8_t h[2];
    CU_TRY(c, cudaMemcpyAsync(&h[0], c->blkstate.p, 1, cudaMemcpyDeviceToHost, c->stream));
    CU_TRY(c, cudaMemcpyAsync(&h[1], c->carry.p, 1, cudaMemcpyDeviceToHost, c->stream));
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    *state_out = (h[0] != ST_P) ? h[0] : h[1];
    return end_call(c);
}

int b200sa_shard_classify(b200sa_ctx *c, const uint8_t *d_shard, uint64_t len, int prev_char, int next_char,
                          int tail_carry, uint32_t *d_stype_words, uint32_t *d_lms_words, uint32_t *d_lmspos,
                          uint64_t cap_lms, uint64_t *hist768, uint64_t *m_out, void *stream) {
    if (!c || !d_shard || len < 1 || len > B200SA_MAX_N || prev_char > 255 || next_char > 255) return B200SA_ERR_BAD_ARG;
    if (next_char >= 0 && tail_carry != (int)ST_L && tail_carry != (int)ST_S) return B200SA_ERR_BAD_ARG;
    if (((uintptr_t)d_shard & 15) != 0) { c->last_error = "shard pointer must be 16-byte aligned"; return B200SA_ERR_BAD_ARG; }
    CU_TRY(c, cudaSetDevice(c->device));
    begin_call(c, stream);
    uint32_t m = 0;
    ShardEdge edge{next_char, prev_char, next_char >= 0 ? (uint32_t)tail_carry : ST_L};
    TRY(classify_dev(c, d_shard, len, &m, edge));
    uint64_t nw = (len + 31) / 32;
    if (d_stype_words) CU_TRY(c, cudaMemcpyAsync(d_stype_words, c->stype.p, nw * 4, cudaMemcpyDeviceToDevice, c->stream));
    if (d_lms_words) CU_TRY(c, cudaMemcpyAsync(d_lms_words, c->lmsb.p, nw * 4, cudaMemcpyDeviceToDevice, c->stream));
    if (d_lmspos && m > 0) {
        uint64_t k = m < cap_lms ? m : cap_lms;
        CU_TRY(c, cudaMemcpyAsync(d_lmspos, c->lmspos.p, k * 4, cudaMemcpyDeviceToDevice, c->stream));
    }
    if (hist768) {
        uint32_t h32[768];
        CU_TRY(c, cudaMemcpyAsync(h32, ptr<uint32_t>(c->tables) + T_HIST, sizeof h32, cudaMemcpyDeviceToHost, c->stream));
        CU_TRY(c, cudaStreamSynchronize(c->stream));
        for (int i = 0; i < 768; i++) hist768[i] = h32[i];
    } else {
        CU_TRY(c, cudaStreamSynchronize(c->stream));
    }
    if (m_out) *m_out = m;
    return end_call(c);
}

// ------------------------------------------------------------ generalized SA / LCP intervals (SURVEY 8f-3, 8f-4)
int b200sa_doc_ids_dev(b200sa_ctx *c, const uint32_t *d_pos, uint64_t count, const uint32_t *d_doc_starts,
                       uint32_t ndocs, uint32_t *d_doc, uint32_t *d_off, void *stream) {
    if (!c || ndocs < 1 || !d_doc_starts || (count > 0 && (!d_pos || !d_doc || !d_off))) return B200SA_ERR_BAD_ARG;
    CU_TRY(c, cudaSetDevice(c->device));
    begin_call(c, stream);
    if (count) LAUNCH(c, k_doc_ids, cdiv(count, BLK), d_pos, count, d_doc_starts, ndocs, d_doc, d_off);
    CU_TRY(c, cudaGetLastError());
    return end_call(c);
}

// Minima of d_lcp over blocks of 32^k entries (in c->qbuf), shared by every k_ansv launch on d_lcp.
static int ansv_levels(b200sa_ctx *c, const uint32_t *d_lcp, uint64_t n, AnsvLevels *L) {
    memset(L, 0, sizeof *L);
    L->lv[0] = d_lcp; L->cnt[0] = n; L->nlev = 1;
    uint64_t total = 0;
    for (uint64_t k = (n + 31) / 32; ; k = (k + 31) / 32) { total += k; if (k <= 32) break; }
    TRY(ensure(c, c->qbuf, (total + 64) * 4));
    uint32_t *lvbuf = ptr<uint32_t>(c->qbuf);
    uint64_t cnt = n;
    while (cnt > 32 && L->nlev < 8) {
        uint64_t nxt = (cnt + 31) / 32;
        LAUNCH(c, k_min32, cdiv(nxt, BLK), L->lv[L->nlev - 1], cnt, lvbuf);
        L->lv[L->nlev] = lvbuf; L->cnt[L->nlev] = nxt; L->nlev++;
        lvbuf += nxt;
        cnt = nxt;
    }
    return B200SA_OK;
}

int b200sa_lcp_intervals_dev(b200sa_ctx *c, const uint32_t *d_lcp, uint64_t n, uint32_t *d_psv, uint32_t *d_nsv,
                             void *stream) {
    if (!c || (n > 0 && (!d_lcp || !d_psv || !d_nsv))) return B200SA_ERR_BAD_ARG;
    if (n > B200SA_MAX_N) return B200SA_ERR_TOO_LARGE;
    CU_TRY(c, cudaSetDevice(c->device));
    begin_call(c, stream);
    if (n == 0) return end_call(c);
    AnsvLevels L;
    TRY(ansv_levels(c, d_lcp, n, &L));
    LAUNCH(c, k_ansv<true>, cdiv(n, BLK), L, n, d_psv, d_nsv);
    CU_TRY(c, cudaGetLastError());
    return end_call(c);
}

// ------------------------------------------------------------ suffix tree (SURVEY 8f-5, tree.cuh)
// Node arrays of the tree of an n-byte text from its SA and LCP on the device; *count = nodes.
// Scratch: p0 psv, p1 nsv, g0 pse, g1 head -> node id, rank e / base, v0 v1 k32b isa the sort.
static int tree_dev(b200sa_ctx *c, uint64_t n, const uint32_t *d_sa, const uint32_t *d_lcp, const b200sa_tree *o,
                    uint64_t *count) {
    if (n <= 1) {
        // root (and the leaf of suffix 0): no launches, six tiny copies through the pinned words
        static const uint32_t one[6][2] = {{TREE_NONE, 0}, {0, 1}, {0, 0}, {1, 1}, {2, 2}, {1, 0}};
        uint32_t *const dst[6] = {o->parent, o->depth, o->lo, o->hi, o->end, o->nchildren};
        for (int f = 0; f < 6; f++) {
            c->h_pin[2 * f] = one[f][0];
            c->h_pin[2 * f + 1] = one[f][1];
        }
        if (n == 0) { c->h_pin[6] = 0; c->h_pin[8] = 1; c->h_pin[10] = 0; }      // hi, end, nchildren of a lone root
        for (int f = 0; f < 6; f++)
            CU_TRY(c, cudaMemcpyAsync(dst[f], c->h_pin + 2 * f, (n + 1) * 4, cudaMemcpyHostToDevice, c->stream));
        CU_TRY(c, cudaStreamSynchronize(c->stream));
        *count = n + 1;
        return B200SA_OK;
    }
    uint32_t n32 = (uint32_t)n;
    TRY(ensure(c, c->p0, n * 4));
    TRY(ensure(c, c->p1, n * 4));
    TRY(ensure(c, c->g0, n * 4));
    TRY(ensure(c, c->g1, n * 4));
    TRY(ensure(c, c->rank, (n + 1) * 4));
    TRY(ensure(c, c->v0, n * 4));
    TRY(ensure(c, c->v1, n * 4));
    TRY(ensure(c, c->k32b, n * 4));
    TRY(ensure(c, c->isa, n * 4));
    TRY(ensure(c, c->small, 4096));
    uint32_t *psv = ptr<uint32_t>(c->p0), *nsv = ptr<uint32_t>(c->p1), *pse = ptr<uint32_t>(c->g0);
    uint32_t *headid = ptr<uint32_t>(c->g1), *base = ptr<uint32_t>(c->rank), *d_m = ptr<uint32_t>(c->small) + 40;
    TRY(mark(c, "tree_ansv"));
    AnsvLevels L;
    TRY(ansv_levels(c, d_lcp, n, &L));
    LAUNCH(c, k_ansv<true>, cdiv(n, BLK), L, n, psv, nsv);
    LAUNCH(c, k_ansv<false>, cdiv(n, BLK), L, n, pse, (uint32_t *)nullptr);
    TRY(mark(c, "tree_heads"));
    TreeIn t{d_sa, d_lcp, psv, nsv, pse, n32};
    TRY((dev_scan<OpSum>(c, InTreeHead{d_sa, d_lcp, psv, pse, n32}, OutTreeHead{psv, ptr<uint32_t>(c->v0), ptr<uint32_t>(c->v1), n32},
                         n, d_m)));
    TRY(read_words(c, d_m, 1));
    uint32_t m = c->h_pin[0];
    TRY(mark(c, "tree_sort"));
    uint32_t *key = ptr<uint32_t>(c->v0), *val = ptr<uint32_t>(c->v1);
    TRY(sort_pairs<uint32_t>(c, key, val, ptr<uint32_t>(c->k32b), ptr<uint32_t>(c->isa), m, bit_length(n - 1),
                             &key, &val));
    TRY(mark(c, "tree_base"));
    CU_TRY(c, cudaMemsetAsync(base, 0, (n + 1) * 4, c->stream));
    if (m) LAUNCH(c, k_tree_bucket_end, cdiv(m, BLK), key, m, base);
    TRY((dev_scan<OpMax>(c, InArray{base}, OutTreeBase{base}, n + 1, nullptr)));
    TRY(mark(c, "tree_nodes"));
    uint64_t nodes = 1 + n + (uint64_t)m;
    TreeOut to{o->parent, o->depth, o->lo, o->hi, o->end, o->nchildren};
    CU_TRY(c, cudaMemsetAsync(o->nchildren, 0, nodes * 4, c->stream));
    if (m) LAUNCH(c, k_tree_internal, cdiv(m, BLK), t, key, val, m, base, headid, to);
    LAUNCH(c, k_tree_link, cdiv(n, BLK), t, base, headid, to);
    TRY(mark(c, "end"));
    CU_TRY(c, cudaGetLastError());
    *count = nodes;
    return B200SA_OK;
}

int b200sa_suffix_tree_dev(b200sa_ctx *c, const uint8_t *d_text, uint64_t n, const uint32_t *d_sa,
                           const uint32_t *d_lcp, const b200sa_tree *d_out, uint64_t *num_nodes, void *stream) {
    if (!c) return B200SA_ERR_BAD_ARG;
    if (n > B200SA_TREE_MAX_N) { c->last_error = "text longer than B200SA_TREE_MAX_N = 2^31-1 bytes"; return B200SA_ERR_TOO_LARGE; }
    if (!d_out || !num_nodes || (n > 0 && (!d_text || !d_sa || !d_lcp)) || !d_out->parent || !d_out->depth ||
        !d_out->lo || !d_out->hi || !d_out->end || !d_out->nchildren)
        return B200SA_ERR_BAD_ARG;
    CU_TRY(c, cudaSetDevice(c->device));
    begin_call(c, stream);
    TRY(tree_dev(c, n, d_sa, d_lcp, d_out, num_nodes));
    return end_call(c);
}

static int host_tree_inner(b200sa_ctx *c, const uint8_t *text, uint64_t n, uint32_t *sa, int sa_given,
                           const b200sa_tree *h, uint64_t *num_nodes) {
    CU_TRY(c, cudaSetDevice(c->device));
    begin_call(c, nullptr);
    memset(&c->stats, 0, sizeof c->stats);
    c->stats.n = n;
    size_t cap = n ? 2 * n : 1;
    TRY(ensure(c, c->tree, 6 * cap * 4));
    uint32_t *tb = ptr<uint32_t>(c->tree);
    b200sa_tree d{tb, tb + cap, tb + 2 * cap, tb + 3 * cap, tb + 4 * cap, tb + 5 * cap};
    const uint32_t *d_sa = nullptr, *d_lcp = nullptr;
    if (n >= 1) {
        TRY(ensure(c, c->text, n));
        TRY(ensure(c, c->sa, n * 4));
        TRY(ensure(c, c->lcp, n * 4));
        TRY(mark(c, "h2d"));
        CU_TRY(c, cudaMemcpyAsync(c->text.p, text, n, cudaMemcpyHostToDevice, c->stream));
        if (sa_given) {
            // SuffixTree::from_suffix_table: the table comes from the caller, lcp_dev checks it; the
            // tree kernels need the LCP intervals of the sorted table, so any other table is rejected
            CU_TRY(c, cudaMemcpyAsync(c->sa.p, sa, n * 4, cudaMemcpyHostToDevice, c->stream));
            TRY(lcp_dev(c, ptr<uint8_t>(c->text), n, ptr<uint32_t>(c->sa), ptr<uint32_t>(c->lcp), false, true));
        } else {
            TRY(build_dev(c, ptr<uint8_t>(c->text), n, ptr<uint32_t>(c->sa)));
            TRY(lcp_dev(c, ptr<uint8_t>(c->text), n, ptr<uint32_t>(c->sa), ptr<uint32_t>(c->lcp), n >= 2));
        }
        d_sa = ptr<uint32_t>(c->sa);
        d_lcp = ptr<uint32_t>(c->lcp);
    }
    uint64_t k = 0;
    TRY(tree_dev(c, n, d_sa, d_lcp, &d, &k));
    TRY(mark(c, "d2h_tree"));
    if (!sa_given && n) CU_TRY(c, cudaMemcpyAsync(sa, c->sa.p, n * 4, cudaMemcpyDeviceToHost, c->stream));
    uint32_t *const src[6] = {d.parent, d.depth, d.lo, d.hi, d.end, d.nchildren};
    uint32_t *const dst[6] = {h->parent, h->depth, h->lo, h->hi, h->end, h->nchildren};
    for (int f = 0; f < 6; f++) CU_TRY(c, cudaMemcpyAsync(dst[f], src[f], k * 4, cudaMemcpyDeviceToHost, c->stream));
    TRY(mark(c, "end"));
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    *num_nodes = k;
    return end_call(c);
}

int b200sa_suffix_tree(b200sa_ctx *c, const uint8_t *text, uint64_t n, uint32_t *sa, int sa_given,
                       const b200sa_tree *h_out, uint64_t *num_nodes) {
    if (!c) return B200SA_ERR_BAD_ARG;
    if (n > B200SA_TREE_MAX_N) { c->last_error = "text longer than B200SA_TREE_MAX_N = 2^31-1 bytes"; return B200SA_ERR_TOO_LARGE; }
    if (!h_out || !num_nodes || (n > 0 && (!text || !sa)) || !h_out->parent || !h_out->depth || !h_out->lo ||
        !h_out->hi || !h_out->end || !h_out->nchildren)
        return B200SA_ERR_BAD_ARG;
    int rc = host_tree_inner(c, text, n, sa, sa_given, h_out, num_nodes);
    if (rc != B200SA_OK) {
        if (c->stream) cudaStreamSynchronize(c->stream);
        cudaGetLastError();
    }
    return rc;
}

// ------------------------------------------------------------ multi-GPU: communicator + sharded LMS sort
#define NCCL_TRY(ctx, expr)                                                                  \
    do {                                                                                     \
        ncclResult_t r__ = (expr);                                                           \
        if (r__ != ncclSuccess) {                                                            \
            char buf__[400];                                                                 \
            snprintf(buf__, sizeof buf__, "%s:%d: %s -> %s", __FILE__, __LINE__, #expr,      \
                     nccl_api().GetErrorString ? nccl_api().GetErrorString(r__) : "nccl error"); \
            (ctx)->last_error = buf__;                                                       \
            return B200SA_ERR_COMM;                                                          \
        }                                                                                    \
    } while (0)

int b200sa_comm_unique_id(uint8_t *id_out) {
    if (!id_out) return B200SA_ERR_BAD_ARG;
    NcclApi &N = nccl_api();
    if (!N.ok) return B200SA_ERR_COMM;
    ncclUniqueId id;
    if (N.GetUniqueId(&id) != ncclSuccess) return B200SA_ERR_COMM;
    memcpy(id_out, id.internal, NCCL_UNIQUE_ID_BYTES);
    return B200SA_OK;
}

int b200sa_comm_init(b200sa_ctx *c, int nranks, int rank, const uint8_t *id128) {
    if (!c || !id128 || nranks < 1 || rank < 0 || rank >= nranks || nranks > 16) return B200SA_ERR_BAD_ARG;
    NcclApi &N = nccl_api();
    if (!N.ok) { c->last_error = N.err; return B200SA_ERR_COMM; }
    CU_TRY(c, cudaSetDevice(c->device));
    if (c->comm && c->comm_owned) N.CommDestroy(c->comm);
    c->comm = nullptr;
    ncclUniqueId id;
    memcpy(id.internal, id128, NCCL_UNIQUE_ID_BYTES);
    NCCL_TRY(c, N.CommInitRank(&c->comm, nranks, id, rank));
    c->comm_owned = true; c->nranks = nranks; c->comm_rank = rank;
    return B200SA_OK;
}

int b200sa_comm_attach(b200sa_ctx *c, void *nccl_comm) {
    if (!c || !nccl_comm) return B200SA_ERR_BAD_ARG;
    NcclApi &N = nccl_api();
    if (!N.ok) { c->last_error = N.err; return B200SA_ERR_COMM; }
    if (c->comm && c->comm_owned) N.CommDestroy(c->comm);
    c->comm = (ncclComm_t)nccl_comm;
    c->comm_owned = false;
    NCCL_TRY(c, N.CommCount(c->comm, &c->nranks));
    NCCL_TRY(c, N.CommUserRank(c->comm, &c->comm_rank));
    if (c->nranks > 16) return B200SA_ERR_BAD_ARG;
    return B200SA_OK;
}

int b200sa_comm_destroy(b200sa_ctx *c) {
    if (!c) return B200SA_ERR_BAD_ARG;
    if (c->comm && c->comm_owned && nccl_api().ok) nccl_api().CommDestroy(c->comm);
    c->comm = nullptr; c->comm_owned = false; c->nranks = 1; c->comm_rank = 0;
    return B200SA_OK;
}

// Collective over the context's communicator (a context without one is a world of 1).
int b200sa_shard_lms_sort(b200sa_ctx *c, const uint8_t *d_shard, uint64_t len, unsigned long long *d_sorted_gpos,
                          uint32_t *d_names, uint64_t cap, b200sa_shard_stats *out, void *stream) {
    if (!c || !d_shard || len < 1 || len > B200SA_MAX_N || !out) return B200SA_ERR_BAD_ARG;
    if (((uintptr_t)d_shard & 15) != 0) { c->last_error = "shard pointer must be 16-byte aligned"; return B200SA_ERR_BAD_ARG; }
    NcclApi &N = nccl_api();
    const int W = c->comm ? c->nranks : 1, R = c->comm ? c->comm_rank : 0;
    if (W > 1 && !N.ok) { c->last_error = N.err; return B200SA_ERR_COMM; }
    CU_TRY(c, cudaSetDevice(c->device));
    begin_call(c, stream);
    memset(out, 0, sizeof *out);
    constexpr int HEAD = 64;                                   // bytes of every shard's head that travel (halo source)
    // ---- small exchange area: per rank {len, first byte, last byte, state, m, distinct} + head bytes
    const size_t REC = 8;                                      // u64 words per rank record
    TRY(ensure(c, c->sh_small, (size_t)W * (REC * 8 + HEAD) * 2 + (size_t)W * W * 8 + 8192));
    unsigned long long *rec_all = ptr<unsigned long long>(c->sh_small);            // [W][REC]
    unsigned long long *rec_mine = rec_all + (size_t)W * REC;                      // [REC]
    uint8_t *heads_all = reinterpret_cast<uint8_t *>(rec_mine + REC);              // [W][HEAD]
    unsigned long long *cntmat = reinterpret_cast<unsigned long long *>(heads_all + (((size_t)W * HEAD + 63) & ~(size_t)63));   // [W][W] send counts
    unsigned long long *cnt_mine = cntmat + (size_t)W * W;                         // [W]
    unsigned long long *h64 = cnt_mine + W;                                        // [768]
    TRY(mark(c, "shard_edges"));
    // record: len, first, last  (+ head bytes)
    {
        unsigned long long h_rec[REC] = {len, 0, 0, 0, 0, 0, 0, cap};        // [7]: output capacity, so that every rank can
                                                                            // see every rank's fit and all fail together
        CU_TRY(c, cudaMemcpyAsync(rec_mine, h_rec, sizeof h_rec, cudaMemcpyHostToDevice, c->stream));
        CU_TRY(c, cudaMemsetAsync(heads_all + (size_t)R * HEAD, 0, HEAD, c->stream));
        CU_TRY(c, cudaMemcpyAsync(heads_all + (size_t)R * HEAD, d_shard, len < HEAD ? len : HEAD, cudaMemcpyDeviceToDevice, c->stream));
        CU_TRY(c, cudaMemcpyAsync(reinterpret_cast<uint8_t *>(rec_mine + 1), d_shard, 1, cudaMemcpyDeviceToDevice, c->stream));
        CU_TRY(c, cudaMemcpyAsync(reinterpret_cast<uint8_t *>(rec_mine + 2), d_shard + len - 1, 1, cudaMemcpyDeviceToDevice, c->stream));
    }
    std::vector<unsigned long long> hrec((size_t)W * REC);
    std::vector<uint8_t> hheads((size_t)W * HEAD);
    auto gather_records = [&]() -> int {
        if (W > 1) {
            NCCL_TRY(c, N.AllGather(rec_mine, rec_all, REC, ncclUint64, c->comm, c->stream));
        } else {
            CU_TRY(c, cudaMemcpyAsync(rec_all, rec_mine, REC * 8, cudaMemcpyDeviceToDevice, c->stream));
        }
        CU_TRY(c, cudaMemcpyAsync(hrec.data(), rec_all, (size_t)W * REC * 8, cudaMemcpyDeviceToHost, c->stream));
        return B200SA_OK;
    };
    TRY(gather_records());
    if (W > 1) NCCL_TRY(c, N.AllGather(heads_all + (size_t)R * HEAD, heads_all, HEAD, ncclUint8, c->comm, c->stream));
    CU_TRY(c, cudaMemcpyAsync(hheads.data(), heads_all, (size_t)W * HEAD, cudaMemcpyDeviceToHost, c->stream));
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    uint64_t lo = 0, n_total = 0;
    for (int r = 0; r < W; r++) { if (r < R) lo += hrec[r * REC]; n_total += hrec[r * REC]; }
    int next_char = -1, prev_char = -1;
    if (R + 1 < W) next_char = (int)(hrec[(R + 1) * REC + 1] & 0xff);
    if (R > 0) prev_char = (int)(hrec[(R - 1) * REC + 2] & 0xff);
    // halo: the bytes that follow this shard, taken from the heads of the following shards
    std::vector<uint8_t> halo;                     // up to HEAD bytes (or everything up to the end of the text)
    for (int r = R + 1; r < W && halo.size() < (size_t)HEAD; r++) {
        uint64_t take = hrec[r * REC] < (uint64_t)HEAD ? hrec[r * REC] : (uint64_t)HEAD;
        halo.insert(halo.end(), hheads.begin() + (size_t)r * HEAD, hheads.begin() + (size_t)r * HEAD + take);
    }
    if (halo.size() > (size_t)HEAD) halo.resize(HEAD);
    // ---- shard state -> tail carries
    TRY(mark(c, "shard_classify"));
    int state = ST_L;
    if (next_char >= 0) {
        uint64_t nw = (len + 31) / 32;
        uint32_t nbc = cdiv(nw, CLS_WORDS);
        TRY(ensure(c, c->blkstate, nbc));
        TRY(ensure(c, c->carry, nbc));
        ShardEdge e0{next_char, -1, ST_P};
        LAUNCH(c, k_cls_block_state, nbc, d_shard, len, ptr<uint8_t>(c->blkstate), e0);
        LAUNCH(c, k_cls_carry, 1, ptr<uint8_t>(c->blkstate), nbc, ptr<uint8_t>(c->carry), (uint32_t)ST_P);
        uint8_t h2[2];
        CU_TRY(c, cudaMemcpyAsync(&h2[0], c->blkstate.p, 1, cudaMemcpyDeviceToHost, c->stream));
        CU_TRY(c, cudaMemcpyAsync(&h2[1], c->carry.p, 1, cudaMemcpyDeviceToHost, c->stream));
        CU_TRY(c, cudaStreamSynchronize(c->stream));
        state = (h2[0] != ST_P) ? h2[0] : h2[1];
    }
    {
        unsigned long long st = (unsigned long long)state;
        CU_TRY(c, cudaMemcpyAsync(rec_mine + 3, &st, 8, cudaMemcpyHostToDevice, c->stream));
        TRY(gather_records());
        CU_TRY(c, cudaStreamSynchronize(c->stream));
    }
    uint32_t tail = ST_L;
    for (int r = R + 1; r < W; r++) if (hrec[r * REC + 3] != ST_P) { tail = (uint32_t)hrec[r * REC + 3]; break; }
    // ---- classification of the shard (fused kernel with halo chars), LMS positions descending
    uint32_t m = 0;
    TRY(classify_fused_dev(c, d_shard, len, &m, ShardEdge{next_char, prev_char, next_char >= 0 ? tail : ST_L}, false));
    // ---- global alphabet: all-reduce of the (byte, type) histogram
    TRY(mark(c, "shard_keys"));
    uint32_t *tab = ptr<uint32_t>(c->tables);
    LAUNCH(c, k_hist_to_u64, 3u, tab + T_HIST, h64, 768u);
    if (W > 1) NCCL_TRY(c, N.AllReduce(h64, h64, 768, ncclUint64, ncclSum, c->comm, c->stream));
    uint32_t *sm = ptr<uint32_t>(c->small);
    LAUNCH(c, k_alpha_from_hist64, 1u, h64, tab + T_CODE, sm + 3);
    TRY(read_words(c, sm + 3, 1));
    const uint32_t sigma = c->h_pin[0] < 2 ? 2u : c->h_pin[0];
    uint32_t kc = 0;
    {
        unsigned __int128 r = 1;
        while (kc < 32 && r * sigma <= ((unsigned __int128)1 << 64)) { r *= sigma; kc++; }
    }
    // ---- window keys of the local LMS suffixes (descending position order)
    TRY(ensure(c, c->sh_a, (size_t)(m + 1) * 8));                 // keys
    TRY(ensure(c, c->sh_b, (size_t)(m + 1) * 4));                 // local positions
    TRY(ensure(c, c->sh_c, (size_t)(m + 1) * 8));                 // keys partitioned by destination
    TRY(ensure(c, c->sh_d, (size_t)(m + 1) * 4));                 // positions partitioned
    TRY(ensure(c, c->flag, (size_t)m + 64 + HEAD));               // destinations (+ halo bytes at the end)
    uint8_t *d_halo = ptr<uint8_t>(c->flag) + (((size_t)m + 15) & ~(size_t)15);
    if (!halo.empty()) CU_TRY(c, cudaMemcpyAsync(d_halo, halo.data(), halo.size(), cudaMemcpyHostToDevice, c->stream));
    ShardWin SW{d_shard, d_halo, tab + T_CODE, len, (uint64_t)halo.size(), sigma, kc};
    uint64_t *K0 = ptr<uint64_t>(c->sh_a), *K1 = ptr<uint64_t>(c->sh_c);
    uint32_t *V0 = ptr<uint32_t>(c->sh_b), *V1 = ptr<uint32_t>(c->sh_d);
    if (m) LAUNCH(c, k_shard_keys, cdiv(m, BLK), SW, ptr<uint32_t>(c->lmsdesc), m, K0, V0);
    // ---- splitters from an all-gathered sample
    TRY(mark(c, "shard_partition"));
    const uint32_t PER = 1024;
    TRY(ensure(c, c->sh_e, (size_t)W * PER * 8 * 2 + (size_t)W * PER * 4 * 2 + 256));
    uint64_t *samp = ptr<uint64_t>(c->sh_e), *samp2 = samp + (size_t)W * PER;
    uint32_t *sv0 = reinterpret_cast<uint32_t *>(samp2 + (size_t)W * PER), *sv1 = sv0 + (size_t)W * PER;
    uint64_t *split = reinterpret_cast<uint64_t *>(sv1 + (size_t)W * PER);
    LAUNCH(c, k_shard_sample, cdiv(PER, BLK), K0, m, PER, samp + (size_t)R * PER);
    if (W > 1) NCCL_TRY(c, N.AllGather(samp + (size_t)R * PER, samp, PER, ncclUint64, c->comm, c->stream));
    {
        uint64_t *ks; uint32_t *vs;
        LAUNCH(c, k_iota, cdiv(W * PER, BLK), sv0, (uint32_t)(W * PER));
        TRY(sort_pairs<uint64_t>(c, samp, sv0, samp2, sv1, (uint64_t)W * PER, 64, &ks, &vs));
        LAUNCH(c, k_shard_splitters, 1u, ks, (uint32_t)(W * PER), (uint32_t)W, split);
    }
    CU_TRY(c, cudaMemsetAsync(cnt_mine, 0, (size_t)W * 8, c->stream));
    uint8_t *dest = ptr<uint8_t>(c->flag);
    if (m) {
        LAUNCH(c, k_shard_dest, cdiv(m, BLK), K0, m, split, (uint32_t)W, dest, cnt_mine);
        TRY(radix_pass(c, DigU8{dest}, MoveKV64{K0, V0, K1, V1}, m));        // stable: descending position inside a destination
    }
    if (W > 1) NCCL_TRY(c, N.AllGather(cnt_mine, cntmat, W, ncclUint64, c->comm, c->stream));
    else CU_TRY(c, cudaMemcpyAsync(cntmat, cnt_mine, 8, cudaMemcpyDeviceToDevice, c->stream));
    std::vector<unsigned long long> hcnt((size_t)W * W);
    CU_TRY(c, cudaMemcpyAsync(hcnt.data(), cntmat, (size_t)W * W * 8, cudaMemcpyDeviceToHost, c->stream));
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    // ---- all-to-all: chunks are received in DESCENDING source rank (larger text positions first)
    TRY(mark(c, "shard_exchange"));
    uint64_t recv_total = 0, m_total = 0;
    std::vector<uint64_t> roff(W + 1, 0), soff(W + 1, 0);
    for (int k = 0; k < W; k++) { int src = W - 1 - k; roff[k + 1] = roff[k] + hcnt[(size_t)src * W + R]; }
    for (int d = 0; d < W; d++) soff[d + 1] = soff[d] + hcnt[(size_t)R * W + d];
    recv_total = roff[W];
    for (int r = 0; r < W; r++) for (int d = 0; d < W; d++) m_total += hcnt[(size_t)r * W + d];
    for (int r = 0; r < W; r++) {                  // the same verdict on every rank: nobody enters the exchange alone
        uint64_t slice = 0;
        for (int q = 0; q < W; q++) slice += hcnt[(size_t)q * W + r];
        if (slice > 0xfffffff0ull) { c->last_error = "more than 2^32 LMS suffixes on one rank"; return B200SA_ERR_TOO_LARGE; }
        if (slice > hrec[r * REC + 7]) {
            char b[160]; snprintf(b, sizeof b, "output capacity of rank %d too small for its slice (%llu entries)", r, (unsigned long long)slice);
            c->last_error = b; return B200SA_ERR_BAD_ARG;
        }
    }
    TRY(ensure(c, c->sh_a, (size_t)(recv_total + 1) * 8));         // received keys (K0 is free after the partition)
    TRY(ensure(c, c->sh_b, (size_t)(recv_total + 1) * 4));         // received local positions
    K0 = ptr<uint64_t>(c->sh_a); V0 = ptr<uint32_t>(c->sh_b);
    if (W > 1) {
        NCCL_TRY(c, N.GroupStart());
        for (int k = 0; k < W; k++) {
            int src = W - 1 - k;
            uint64_t cnt = roff[k + 1] - roff[k];
            if (cnt) {
                NCCL_TRY(c, N.Recv(K0 + roff[k], cnt, ncclUint64, src, c->comm, c->stream));
                NCCL_TRY(c, N.Recv(V0 + roff[k], cnt, ncclUint32, src, c->comm, c->stream));
            }
        }
        for (int d = 0; d < W; d++) {
            uint64_t cnt = soff[d + 1] - soff[d];
            if (cnt) {
                NCCL_TRY(c, N.Send(K1 + soff[d], cnt, ncclUint64, d, c->comm, c->stream));
                NCCL_TRY(c, N.Send(V1 + soff[d], cnt, ncclUint32, d, c->comm, c->stream));
                if (d != R) { out->bytes_sent += (double)cnt * 12.0; }
            }
        }
        NCCL_TRY(c, N.GroupEnd());
    } else if (recv_total) {
        CU_TRY(c, cudaMemcpyAsync(K0, K1, recv_total * 8, cudaMemcpyDeviceToDevice, c->stream));
        CU_TRY(c, cudaMemcpyAsync(V0, V1, recv_total * 4, cudaMemcpyDeviceToDevice, c->stream));
    }
    // ---- local sort of the received slice, global positions, groups, names
    TRY(mark(c, "shard_sort"));
    uint32_t cnt32 = (uint32_t)recv_total;
    TRY(ensure(c, c->sh_c, (size_t)(recv_total + 1) * 8));
    TRY(ensure(c, c->sh_d, (size_t)(recv_total + 1) * 4));
    TRY(ensure(c, c->sh_f, (size_t)(recv_total + 1) * 4));
    uint32_t *I0 = ptr<uint32_t>(c->sh_d), *I1 = ptr<uint32_t>(c->sh_f);
    uint64_t *Ks = K0; uint32_t *Is = I0;
    unsigned long long *chunk_off = cnt_mine;                      // reuse: [W+1] offsets, then [W] lo
    std::vector<unsigned long long> hco((size_t)2 * W + 1);
    for (int k = 0; k <= W; k++) hco[k] = roff[k];
    for (int k = 0; k < W; k++) { int src = W - 1 - k; uint64_t l2 = 0; for (int r = 0; r < src; r++) l2 += hrec[r * REC]; hco[W + 1 + k] = l2; }
    TRY(ensure(c, c->sh_e, (size_t)(2 * W + 1) * 8 + 64));
    chunk_off = ptr<unsigned long long>(c->sh_e);
    CU_TRY(c, cudaMemcpyAsync(chunk_off, hco.data(), hco.size() * 8, cudaMemcpyHostToDevice, c->stream));
    unsigned long long *d_ties = h64;                              // reuse (the histogram is consumed)
    CU_TRY(c, cudaMemsetAsync(d_ties, 0, 16, c->stream));
    if (cnt32) {
        LAUNCH(c, k_iota, cdiv(cnt32, BLK), I0, cnt32);
        int kbits = 64;
        TRY(sort_pairs<uint64_t>(c, K0, I0, ptr<uint64_t>(c->sh_c), I1, cnt32, kbits, &Ks, &Is));
        LAUNCH(c, k_shard_gpos, cdiv(cnt32, BLK), Is, V0, cnt32, chunk_off, chunk_off + W + 1, (uint32_t)W, d_sorted_gpos);
        InShardHead in{Ks, d_sorted_gpos, cnt32, n_total, kc};
        TRY((dev_scan<OpSum>(c, in, OutShardName{in, 0u, d_names, d_ties}, cnt32, sm + 16)));
    } else {
        CU_TRY(c, cudaMemsetAsync(sm + 16, 0, 4, c->stream));
    }
    // ---- name offsets: exclusive prefix of the distinct counts over ranks; ties summed
    TRY(mark(c, "shard_names"));
    CU_TRY(c, cudaMemcpyAsync(reinterpret_cast<uint32_t *>(rec_mine + 5), sm + 16, 4, cudaMemcpyDeviceToDevice, c->stream));
    CU_TRY(c, cudaMemcpyAsync(rec_mine + 6, d_ties, 8, cudaMemcpyDeviceToDevice, c->stream));
    {
        unsigned long long mm = m;
        CU_TRY(c, cudaMemcpyAsync(rec_mine + 4, &mm, 8, cudaMemcpyHostToDevice, c->stream));
    }
    TRY(gather_records());
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    uint64_t name_off = 0, ties = 0;
    for (int r = 0; r < W; r++) { if (r < R) name_off += (uint32_t)hrec[r * REC + 5]; ties += hrec[r * REC + 6]; }
    if (cnt32 && name_off) LAUNCH(c, k_add_u32, cdiv(cnt32, BLK), d_names, cnt32, (uint32_t)name_off);
    TRY(mark(c, "end"));
    CU_TRY(c, cudaGetLastError());
    out->n_total = n_total; out->m_total = m_total; out->m_local = m; out->recv_count = recv_total;
    out->distinct_local = (uint32_t)hrec[R * REC + 5]; out->name_offset = name_off; out->ties_total = ties;
    out->kc = kc; out->lo = lo; out->nranks = (uint32_t)W; out->rank = (uint32_t)R;
    out->bytes_recv = 0;
    for (int k = 0; k < W; k++) { int src = W - 1 - k; if (src != R) out->bytes_recv += (double)(roff[k + 1] - roff[k]) * 12.0; }
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    return end_call(c);
}

// Sharded LCP (SURVEY 8e row 5): text and SA are replicated (broadcast from rank 0 unless the caller
// says they already are), every rank computes Phi and PLCP for ITS text range only, the PLCP ranges
// are all-gathered, every rank turns its rank range into LCP values and the slices are all-gathered.
// Same values as lcp_lens_quadratic (src/table.rs:348-361).
int b200sa_lcp_sharded(b200sa_ctx *c, uint8_t *d_text, uint64_t n, uint32_t *d_sa, uint32_t *d_lcp, int replicated,
                       void *stream) {
    if (!c || (n > 0 && (!d_text || !d_sa || !d_lcp))) return B200SA_ERR_BAD_ARG;
    if (n > B200SA_MAX_N) return B200SA_ERR_TOO_LARGE;
    NcclApi &N = nccl_api();
    const int W = c->comm ? c->nranks : 1, R = c->comm ? c->comm_rank : 0;
    if (W > 1 && !N.ok) { c->last_error = N.err; return B200SA_ERR_COMM; }
    CU_TRY(c, cudaSetDevice(c->device));
    begin_call(c, stream);
    if (n == 0) return end_call(c);
    if (((uintptr_t)d_text & 15) != 0) { c->last_error = "text pointer must be 16-byte aligned"; return B200SA_ERR_BAD_ARG; }
    const uint32_t n32 = (uint32_t)n;
    TRY(mark(c, "lcps_bcast"));
    if (W > 1 && !replicated) {
        NCCL_TRY(c, N.Broadcast(d_text, d_text, n, ncclUint8, 0, c->comm, c->stream));
        NCCL_TRY(c, N.Broadcast(d_sa, d_sa, n, ncclUint32, 0, c->comm, c->stream));
    }
    // ---- every rank: validate the table, pack the text (same steps as the stand-alone b200sa_lcp_dev)
    TRY(mark(c, "lcps_pack"));
    const uint64_t per = ((n + W - 1) / W + 1023) / 1024 * 1024;       // positions (and ranks) per GPU
    TRY(ensure(c, c->isa, (size_t)W * per * 4));
    TRY(ensure(c, c->small, 4096));
    TRY(ensure(c, c->tables, T_END * 4));
    uint32_t *tab = ptr<uint32_t>(c->tables), *sm = ptr<uint32_t>(c->small);
    {
        uint64_t nwv = (n + 31) / 32;
        uint32_t *seen = ptr<uint32_t>(c->isa), *bad = sm + 12;
        CU_TRY(c, cudaMemsetAsync(seen, 0, nwv * 4, c->stream));
        CU_TRY(c, cudaMemsetAsync(bad, 0, 4, c->stream));
        CU_TRY(c, cudaMemsetAsync(bad + 1, 0, 4, c->stream));
        LAUNCH(c, k_sa_validate, cdiv(cdiv(n, 4), BLK), d_sa, n32, seen, bad);
        LAUNCH(c, k_sa_validate_count, 592u, seen, n32, bad + 1);
        LAUNCH(c, k_sa_validate_verdict, 1u, bad + 1, n32, bad);
        CU_TRY(c, cudaMemsetAsync(tab + T_HIST, 0, 256 * 4, c->stream));
        uint32_t hb = cdiv(n, BLK * 64);
        if (hb > 1184) hb = 1184;
        LAUNCH(c, k_byte_hist, hb, d_text, n, tab + T_HIST);
        LAUNCH(c, k_alpha_from_hist, 1, tab + T_HIST, tab + T_CODE, tab + T_ALPHA, sm + 3);
        TRY(read_words(c, sm, 16));
        if (c->h_pin[12] != 0) {      // identical on every rank: all fail together
            c->last_error = "table is not a permutation of 0..n-1 (index out of range or repeated)";
            return B200SA_ERR_BAD_ARG;
        }
        TRY(pack_text(c, d_text, n, c->h_pin[3]));
    }
    // ---- every rank: is the table the suffix array?  Phi / PLCP is only valid on the sorted table.
    // Every rank holds the whole table, so all reach the same verdict; on a permutation that is not
    // sorted each rank computes the whole array with the reference's per-pair compare, and no rank
    // enters the collectives below.
    TRY(mark(c, "lcp_sorted"));
    {
        bool sorted = false;
        TRY(sa_is_sorted(c, d_text, n, d_sa, ptr<uint32_t>(c->isa), &sorted));
        if (!sorted) {
            TRY(mark(c, "lcp_unsorted"));
            lcp_direct_launch(c, n32, d_sa, d_lcp, n32, sm + 8);
            TRY(mark(c, "end"));
            CU_TRY(c, cudaGetLastError());
            CU_TRY(c, cudaStreamSynchronize(c->stream));
            return end_call(c);
        }
    }
    // ---- Phi and PLCP of this rank's text range
    TRY(mark(c, "lcps_plcp"));
    const uint64_t lo = (uint64_t)R * per, hi = (lo + per < n) ? lo + per : (lo < n ? n : lo);
    uint32_t *phi = ptr<uint32_t>(c->isa);
    uint32_t nchunk = cdiv(n, LCP_CHUNK);
    TRY(ensure(c, c->plcp_samp, (size_t)nchunk * 4));
    uint32_t *samp = ptr<uint32_t>(c->plcp_samp);
    if (hi > lo) {
        LAUNCH(c, k_phi_range, cdiv(n, BLK), d_sa, n32, (uint32_t)lo, (uint32_t)hi, phi);
        uint64_t len = hi - lo;
        uint32_t chunks = cdiv(len, LCP_CHUNK);
        uint32_t pg = cdiv(chunks, BLK), sg = cdiv(cdiv(chunks, 32), BLK);
        uint64_t toff_s = lo / (32ull * LCP_CHUNK), toff_p = lo / LCP_CHUNK;
        if (c->bits == 2) LAUNCH(c, (k_plcp_samples<2>), sg, c->ptext, n32, phi, samp, toff_s, hi);
        else if (c->bits == 4) LAUNCH(c, (k_plcp_samples<4>), sg, c->ptext, n32, phi, samp, toff_s, hi);
        else LAUNCH(c, (k_plcp_samples<8>), sg, c->ptext, n32, phi, samp, toff_s, hi);
        if (c->bits == 2) LAUNCH(c, (k_plcp<2>), pg, c->ptext, n32, phi, samp, toff_p, hi);
        else if (c->bits == 4) LAUNCH(c, (k_plcp<4>), pg, c->ptext, n32, phi, samp, toff_p, hi);
        else LAUNCH(c, (k_plcp<8>), pg, c->ptext, n32, phi, samp, toff_p, hi);
    }
    TRY(mark(c, "lcps_allgather_plcp"));
    if (W > 1) NCCL_TRY(c, N.AllGather(phi + lo, phi, per, ncclUint32, c->comm, c->stream));
    // ---- LCP of this rank's RANK range, then the slices to everybody
    TRY(mark(c, "lcps_gather"));
    TRY(ensure(c, c->phik, (size_t)W * per * 4));
    uint32_t *slices = ptr<uint32_t>(c->phik);
    if (hi > lo) LAUNCH(c, k_lcp_gather_range, cdiv(hi - lo, BLK), d_sa, phi, (uint32_t)lo, (uint32_t)hi, slices + lo);
    TRY(mark(c, "lcps_allgather_lcp"));
    if (W > 1) NCCL_TRY(c, N.AllGather(slices + lo, slices, per, ncclUint32, c->comm, c->stream));
    CU_TRY(c, cudaMemcpyAsync(d_lcp, slices, n * 4, cudaMemcpyDeviceToDevice, c->stream));
    TRY(mark(c, "end"));
    CU_TRY(c, cudaGetLastError());
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    return end_call(c);
}

// ------------------------------------------------------------ test hooks
int b200sa_test_classify(b200sa_ctx *c, const uint8_t *text, uint64_t n, uint32_t *stype_words, uint32_t *lms_words,
                         uint32_t *hist768, uint32_t *lmspos, uint64_t cap_lms, uint64_t *m_out) {
    if (!c || !text || n < 1 || n > B200SA_MAX_N) return B200SA_ERR_BAD_ARG;
    CU_TRY(c, cudaSetDevice(c->device));
    begin_call(c, nullptr);
    TRY(ensure(c, c->text, n));
    CU_TRY(c, cudaMemcpyAsync(c->text.p, text, n, cudaMemcpyHostToDevice, c->stream));
    uint32_t m = 0;
    TRY(classify_dev(c, ptr<uint8_t>(c->text), n, &m));
    uint64_t nw = (n + 31) / 32;
    if (stype_words) CU_TRY(c, cudaMemcpyAsync(stype_words, c->stype.p, nw * 4, cudaMemcpyDeviceToHost, c->stream));
    if (lms_words) CU_TRY(c, cudaMemcpyAsync(lms_words, c->lmsb.p, nw * 4, cudaMemcpyDeviceToHost, c->stream));
    if (hist768) CU_TRY(c, cudaMemcpyAsync(hist768, ptr<uint32_t>(c->tables) + T_HIST, 768 * 4, cudaMemcpyDeviceToHost, c->stream));
    if (lmspos && m > 0) {
        uint64_t k = m < cap_lms ? m : cap_lms;
        CU_TRY(c, cudaMemcpyAsync(lmspos, c->lmspos.p, k * 4, cudaMemcpyDeviceToHost, c->stream));
    }
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    if (m_out) *m_out = m;
    return end_call(c);
}

int b200sa_test_classify_fused(b200sa_ctx *c, const uint8_t *text, uint64_t n, uint32_t *stype_words, uint32_t *lms_words,
                               uint32_t *hist768, uint32_t *lmspos_desc, uint64_t cap_lms, uint64_t *m_out) {
    if (!c || !text || n < 1 || n > B200SA_MAX_N) return B200SA_ERR_BAD_ARG;
    CU_TRY(c, cudaSetDevice(c->device));
    begin_call(c, nullptr);
    TRY(ensure(c, c->text, n));
    CU_TRY(c, cudaMemcpyAsync(c->text.p, text, n, cudaMemcpyHostToDevice, c->stream));
    uint32_t m = 0;
    TRY(classify_fused_dev(c, ptr<uint8_t>(c->text), n, &m));
    uint64_t nw = (n + 31) / 32;
    if (stype_words) CU_TRY(c, cudaMemcpyAsync(stype_words, c->stype.p, nw * 4, cudaMemcpyDeviceToHost, c->stream));
    if (lms_words) CU_TRY(c, cudaMemcpyAsync(lms_words, c->lmsb.p, nw * 4, cudaMemcpyDeviceToHost, c->stream));
    if (hist768) CU_TRY(c, cudaMemcpyAsync(hist768, ptr<uint32_t>(c->tables) + T_HIST, 768 * 4, cudaMemcpyDeviceToHost, c->stream));
    if (lmspos_desc && m > 0) {
        uint64_t k = m < cap_lms ? m : cap_lms;
        CU_TRY(c, cudaMemcpyAsync(lmspos_desc, c->lmsdesc.p, k * 4, cudaMemcpyDeviceToHost, c->stream));
    }
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    if (m_out) *m_out = m;
    return end_call(c);
}

int b200sa_test_scan(b200sa_ctx *c, const uint32_t *in, uint64_t n, int op, uint32_t *out_excl, uint32_t *total) {
    if (!c || (n > 0 && (!in || !out_excl))) return B200SA_ERR_BAD_ARG;
    CU_TRY(c, cudaSetDevice(c->device));
    begin_call(c, nullptr);
    TRY(ensure(c, c->v0, n * 4));
    TRY(ensure(c, c->v1, n * 4));
    TRY(ensure(c, c->small, 4096));
    CU_TRY(c, cudaMemcpyAsync(c->v0.p, in, n * 4, cudaMemcpyHostToDevice, c->stream));
    uint32_t *d_tot = ptr<uint32_t>(c->small);
    if (op == 0) TRY((dev_scan<OpSum>(c, InArray{ptr<uint32_t>(c->v0)}, OutStoreExcl{ptr<uint32_t>(c->v1)}, n, d_tot)));
    else TRY((dev_scan<OpMax>(c, InArray{ptr<uint32_t>(c->v0)}, OutStoreExcl{ptr<uint32_t>(c->v1)}, n, d_tot)));
    if (n) CU_TRY(c, cudaMemcpyAsync(out_excl, c->v1.p, n * 4, cudaMemcpyDeviceToHost, c->stream));
    TRY(read_words(c, d_tot, 1));
    if (total) *total = c->h_pin[0];
    return end_call(c);
}

int b200sa_test_sort_pairs32(b200sa_ctx *c, uint32_t *keys, uint32_t *vals, uint64_t n, int bits) {
    return test_sort<uint32_t>(c, keys, vals, n, bits);
}
int b200sa_test_sort_pairs64(b200sa_ctx *c, uint64_t *keys, uint32_t *vals, uint64_t n, int bits) {
    return test_sort<uint64_t>(c, keys, vals, n, bits);
}

int b200sa_test_reduced_sa(b200sa_ctx *c, const uint32_t *R, uint64_t m, uint32_t names, uint32_t *sa_out,
                           uint32_t *rounds_out) {
    if (!c || m < 1 || m > 0x7FFFFFFFull || !R || !sa_out) return B200SA_ERR_BAD_ARG;
    CU_TRY(c, cudaSetDevice(c->device));
    begin_call(c, nullptr);
    TRY(ensure(c, c->reduced, m * 4));
    CU_TRY(c, cudaMemcpyAsync(c->reduced.p, R, m * 4, cudaMemcpyHostToDevice, c->stream));
    uint32_t rounds = 0;
    TRY(reduced_sa(c, ptr<uint32_t>(c->reduced), (uint32_t)m, names, &rounds));
    CU_TRY(c, cudaMemcpyAsync(sa_out, c->sa_r.p, m * 4, cudaMemcpyDeviceToHost, c->stream));
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    if (rounds_out) *rounds_out = rounds;
    return end_call(c);
}

int64_t b200sa_debug_fetch(b200sa_ctx *c, int which, void *out, uint64_t cap) {
    if (!c || !out) return B200SA_ERR_BAD_ARG;
    if (cudaSetDevice(c->device) != cudaSuccess) return B200SA_ERR_CUDA;
    const void *src = nullptr;
    uint64_t count = 0;
    switch (which) {
        case 0: src = c->lmspos.p; count = c->last_m; break;
        case 1: src = c->sorted.p; count = c->last_m; break;
        case 2: src = c->reduced.p; count = c->last_m; break;
        case 3: src = c->sa_r.p; count = c->last_m; break;
        case 4: src = c->lmslist.p; count = c->last_m; break;
        case 5: src = c->small.p ? (const void *)(ptr<uint32_t>(c->small) + 32) : nullptr; count = 10; break;
        case 6: src = c->tables.p; count = T_HIST; break;
        case 7: src = c->steplog.p; count = c->steplog.p ? 16384 : 0; break;     // u64 records viewed as u32 pairs
        default: return B200SA_ERR_BAD_ARG;
    }
    if (!src) return 0;
    uint64_t k = count < cap ? count : cap;
    if (k && cudaMemcpy(out, src, k * 4, cudaMemcpyDeviceToHost) != cudaSuccess) return B200SA_ERR_CUDA;
    return (int64_t)count;
}

}  // extern "C"

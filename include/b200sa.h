/*
 * b200sa.h -- C-ABI of the B200-native suffix-array / LCP construction engine.
 *
 * Drop-in boundary for the construction hot path of BurntSushi/suffix
 * (reference: /root/reference/src/table.rs).  The reference has no FFI of its
 * own; the seam is the two private calls made by its public API:
 *
 *   SuffixTable::new      -> sais_table(&text)            src/table.rs:83, :378-386
 *   SuffixTable::lcp_lens -> lcp_lens_quadratic(text,sa)  src/table.rs:135, :348-361
 *
 * Every entry point takes plain pointers and sizes (no torch / C++ types).
 * Caller owns every buffer passed in; the library never retains host
 * pointers after return.  Device workspace is owned by the context and is
 * reused across calls.  A context is NOT thread-safe; distinct contexts are.
 * There is NO CPU fallback: without a usable CUDA device every call returns
 * B200SA_ERR_NO_DEVICE / B200SA_ERR_CUDA.
 *
 * Suffix indices are byte offsets stored as u32 (reference: src/table.rs:64-66).
 * The reference accepts n <= 2^32-1 (src/table.rs:380); this library accepts
 * n <= B200SA_MAX_N = 2^32-4096 (grid index arithmetic is done in u32 with
 * tile-sized slack) and returns B200SA_ERR_TOO_LARGE above that.  Measured up
 * to n = 3*10^9 (profiles/r01_big_configs.jsonl).
 */
#ifndef B200SA_H
#define B200SA_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct b200sa_ctx b200sa_ctx;

#define B200SA_MAX_N 0xFFFFF000ull

enum {
    B200SA_OK            =  0,
    B200SA_ERR_BAD_ARG   = -1,  /* null pointer / bad size / (lcp) table not a permutation of 0..n-1 */
    B200SA_ERR_TOO_LARGE = -2,  /* n > B200SA_MAX_N (reference panics above 2^32-1, src/table.rs:380) */
    B200SA_ERR_NO_DEVICE = -3,
    B200SA_ERR_OOM       = -4,
    B200SA_ERR_CUDA      = -5,
    B200SA_ERR_INTERNAL  = -6,  /* device-side invariant violated                 */
    B200SA_ERR_COMM      = -7   /* NCCL missing or a collective failed            */
};

/* Context: binds a CUDA device, one stream, the device workspace. */
int  b200sa_ctx_create(int device, b200sa_ctx **out);
void b200sa_ctx_destroy(b200sa_ctx *ctx);

/* ---- host-buffer entry points (what a Rust/C++ SuffixTable binds) ---- */

/* Replaces `sais_table(text) -> Vec<u32>` (src/table.rs:378-386), the body of
 * SuffixTable::new (src/table.rs:78-85).  text: n bytes (any bytes; UTF-8 is
 * handled at byte level exactly like the reference's `Utf8` wrapper,
 * src/table.rs:778-800).  sa_out: n u32, caller-allocated.  n==0 and n==1
 * succeed without launching (src/table.rs:395-402). */
int b200sa_build(b200sa_ctx *ctx, const uint8_t *text, uint64_t n, uint32_t *sa_out);

/* Replaces `lcp_lens_quadratic(text, table) -> Vec<u32>` (src/table.rs:348-361)
 * as called by SuffixTable::lcp_lens (src/table.rs:130-138):
 * lcp[0]=0, lcp[i]=|common byte prefix of suffix sa[i-1], suffix sa[i]|.
 * `sa` is checked to be a permutation of 0..n-1 (B200SA_ERR_BAD_ARG otherwise; the
 * reference would panic on an out-of-range index, src/table.rs:356-358).  Any permutation
 * gives lcp_lens_quadratic's array; which path computes it:
 *   - every pair first goes through a direct compare capped at 256 chars (when the text
 *     packs to <= 16 symbols or is <= 32 MiB); if no pair reaches the cap, that is the result;
 *   - otherwise the table is checked to be THE suffix array of the text (one inverse scatter
 *     and one pass over the ranks, phase "lcp_sorted"); the suffix array takes the linear
 *     Phi / PLCP path (Kasai), which is only valid on the sorted table;
 *   - any other permutation (phase "lcp_unsorted") gets the reference's per-pair compare with
 *     no cap: quadratic in the LCP values, like the reference, so slow on repetitive text.
 * b200sa_lcp_dev and b200sa_lcp_sharded follow the same rules; the fused b200sa_build_lcp*
 * built their table themselves and skip the check. */
int b200sa_lcp(b200sa_ctx *ctx, const uint8_t *text, uint64_t n,
               const uint32_t *sa, uint32_t *lcp_out);

/* new + lcp_lens in one call; text and SA stay device-resident in between. */
int b200sa_build_lcp(b200sa_ctx *ctx, const uint8_t *text, uint64_t n,
                     uint32_t *sa_out, uint32_t *lcp_out);

/* ---- device-resident twins (PCIe-free; used by bench.py's `value`) ----
 * d_* are device pointers on the context's device; `stream` is a
 * cudaStream_t (NULL = the context's own stream).  The calls enqueue work and
 * synchronise the stream only where the pipeline must read sizes back. */
int b200sa_build_dev(b200sa_ctx *ctx, const uint8_t *d_text, uint64_t n,
                     uint32_t *d_sa, void *stream);
int b200sa_lcp_dev(b200sa_ctx *ctx, const uint8_t *d_text, uint64_t n,
                   const uint32_t *d_sa, uint32_t *d_lcp, void *stream);
/* new + lcp_lens in one device-resident call (the packed text of the build is
 * reused by the LCP kernels instead of being rebuilt). */
int b200sa_build_lcp_dev(b200sa_ctx *ctx, const uint8_t *d_text, uint64_t n,
                         uint32_t *d_sa, uint32_t *d_lcp, void *stream);

/* ---- batched queries over a device-resident index (SURVEY.md 8f-1) ----
 * Replaces SuffixTable::positions (src/table.rs:223-259) for a batch: query q
 * is bytes [q_off[q], q_off[q+1]) of d_queries; writes the SA range
 * [start[q], end[q]) whose entries are the match positions (SA order, as the
 * reference returns them).  d_sa is trusted like SuffixTable::from_parts (not checked):
 * on any permutation of 0..n-1 the result is what the reference's two binary searches
 * return over that table. */
int b200sa_positions_dev(b200sa_ctx *ctx, const uint8_t *d_text, uint64_t n,
                         const uint32_t *d_sa, const uint8_t *d_queries,
                         const uint64_t *d_q_off, uint32_t nq,
                         uint32_t *d_start, uint32_t *d_end, void *stream);

/* ---- multi-GPU shards (SURVEY.md 8e; BASELINE config 5) ----
 * Type classification + LMS flags + (byte,type) histogram of ONE contiguous
 * shard text[lo,hi) of a longer text, one shard per GPU/process; the caller
 * (suffix_b200/sharded.py, torch.distributed over NCCL) exchanges the tiny
 * summaries between the two calls.  Replaces SuffixTypes::compute
 * (src/table.rs:592-615) and Bins::find_sizes (:686-704) for sharded input.
 *
 * 1. b200sa_shard_summary: *state_out = type of the shard's FIRST position as
 *    far as the shard (plus next_char = T[hi], or -1 at the end of the text)
 *    determines it: 0 Descending(L), 1 Ascending(S), 2 undetermined (every
 *    char up to and including next_char is equal).
 * 2. all-gather the states; tail_carry of shard r = first state != 2 among the
 *    shards after r.
 * 3. b200sa_shard_classify with prev_char = T[lo-1] (-1 for the first shard),
 *    next_char, tail_carry: S-type and LMS bitmaps (bit i&31 of word i>>5,
 *    shard-local positions), shard-local LMS positions (ascending), the
 *    768-bin histogram [0,256) L, [256,512) S-non-LMS, [512,768) LMS (host,
 *    u64, to be all-reduced) and the number of LMS positions.
 * d_shard must be 16-byte aligned. */
int b200sa_shard_summary(b200sa_ctx *ctx, const uint8_t *d_shard, uint64_t len, int next_char,
                         int *state_out, void *stream);
int b200sa_shard_classify(b200sa_ctx *ctx, const uint8_t *d_shard, uint64_t len, int prev_char, int next_char,
                          int tail_carry, uint32_t *d_stype_words, uint32_t *d_lms_words,
                          uint32_t *d_lmspos, uint64_t cap_lms, uint64_t *hist768, uint64_t *m_out, void *stream);

/* ---- generalized suffix array (SURVEY.md 8f-3; reference README.md:60-74, TODO:13-18) ----
 * The reference's own recipe: append the documents with a separator byte that occurs in none
 * of them, remember where each starts, build ONE SuffixTable, and map a match position back
 * to its document with a binary search.  This entry point does that mapping for a batch of
 * positions on the device: doc_starts[0..ndocs) ascending (doc_starts[0] = 0), a position p
 * belongs to the last document d with doc_starts[d] <= p; d_off = p - doc_starts[d].
 * (suffix_b200.GeneralizedSuffixTable is the host-side wrapper.) */
int b200sa_doc_ids_dev(b200sa_ctx *ctx, const uint32_t *d_pos, uint64_t count,
                       const uint32_t *d_doc_starts, uint32_t ndocs,
                       uint32_t *d_doc, uint32_t *d_off, void *stream);

/* ---- LCP-interval tree (SURVEY.md 8f-4; reference suffix_tree/src/lib.rs:392-505) ----
 * The internal nodes of the suffix tree the reference builds serially from SA + LCP are the
 * LCP intervals.  For every rank i: d_psv[i] = largest j < i with lcp[j] < lcp[i]
 * (0xFFFFFFFF if none), d_nsv[i] = smallest j > i with lcp[j] < lcp[i] (n if none); the
 * node that owns the boundary between suffixes i-1 and i is the interval
 * [psv[i], nsv[i]) of string depth lcp[i] (all-nearest-smaller-values over block minima). */
int b200sa_lcp_intervals_dev(b200sa_ctx *ctx, const uint32_t *d_lcp, uint64_t n,
                             uint32_t *d_psv, uint32_t *d_nsv, void *stream);

/* ---- suffix tree (SURVEY.md 8f-5; reference suffix_tree/src/lib.rs) ----
 * The tree the reference's SuffixTree::new / from_suffix_table builds, as structure-of-arrays
 * indexed by preorder id (children in first-byte order = the reference's preorder()):
 *   parent     parent id; 0xFFFFFFFF for the root (id 0)
 *   depth      string depth (length of the path label from the root)
 *   lo, hi     the node's suffixes below it are table[lo, hi) (the root: [0, n))
 *   end        one past the last id of its subtree; children of u are u+1, then end[c]
 *              repeatedly while < end[u]
 *   nchildren  number of children
 * The node's label is text[sa[lo] + depth[parent], sa[lo] + depth).  Like the reference there
 * is no sentinel: a node has a terminal iff depth == n - sa[lo] (suffix sa[lo]), or it is the
 * root (suffix n, empty label); such a leaf may still have children, when its suffix is a
 * prefix of the next one.  There are at most max(2n, 1) nodes.
 * Node ids are u32, so n <= B200SA_TREE_MAX_N; above it both entry points return
 * B200SA_ERR_TOO_LARGE before touching any pointer. */
#define B200SA_TREE_MAX_N 0x7FFFFFFFull
typedef struct {
    uint32_t *parent, *depth, *lo, *hi, *end, *nchildren;
} b200sa_tree;

/* Device-resident construction: d_sa and d_lcp (n u32 each, LCP as lcp_lens) are trusted like
 * SuffixTable::from_parts: they must be the table and LCP array of the n bytes at d_text (the
 * tree is built from them alone; d_text names the text they index).  The six arrays of d_out
 * are device buffers of max(2n, 1) entries; *num_nodes gets the exact node count (one small
 * device-to-host read).  n = 0 and n = 1 launch no kernels. */
int b200sa_suffix_tree_dev(b200sa_ctx *ctx, const uint8_t *d_text, uint64_t n, const uint32_t *d_sa,
                           const uint32_t *d_lcp, const b200sa_tree *d_out, uint64_t *num_nodes, void *stream);

/* Host twin; the six arrays of h_out are host buffers of max(2n, 1) entries.
 *   sa_given == 0: SuffixTree::new -- SA and LCP are built on the device and the SA is written
 *                  to sa[0..n) (labels and terminals need it);
 *   sa_given != 0: SuffixTree::from_suffix_table -- sa[0..n) is read and checked to be THE
 *                  suffix array of the text: a permutation of 0..n-1 in suffix order
 *                  (B200SA_ERR_BAD_ARG otherwise, with b200sa_last_error saying which; the
 *                  tree kernels need the LCP intervals of the sorted table, and the
 *                  reference's construction asserts on other tables), the LCP is computed
 *                  as b200sa_lcp does.
 * The LCP array stays on the device. */
int b200sa_suffix_tree(b200sa_ctx *ctx, const uint8_t *text, uint64_t n, uint32_t *sa, int sa_given,
                       const b200sa_tree *h_out, uint64_t *num_nodes);

/* ---- multi-GPU: communicator + sharded LMS-suffix sort (SURVEY.md 8e, config 5) ----
 * One process (or thread) and one context per GPU.  NCCL is resolved at run time
 * (the copy already loaded in the process, else libnccl.so.2); the single-GPU entry
 * points never touch it.  Either let the library create the communicator --
 * rank 0 calls b200sa_comm_unique_id, the application hands the 128 bytes to every
 * rank (MPI, torch.distributed, a file), every rank calls b200sa_comm_init -- or
 * attach an ncclComm_t the application already owns (same NCCL instance).
 *
 * b200sa_shard_lms_sort (collective): rank r passes its contiguous shard of the
 * text (rank order = text order; 16-byte aligned device pointer).  The shards are
 * classified (types, LMS positions; halo chars and carries exchanged), then the
 * LMS suffixes of the WHOLE text are ordered by their first kc characters (64-bit
 * window keys, zero-padded past the end of the text) with one sample-sort
 * exchange: rank r ends up with the r-th slice of the global order.
 *   d_sorted_gpos[i]  global text position of the i-th LMS suffix of this slice
 *   d_names[i]        dense global rank of its window (equal windows share a name)
 *   out->ties_total   members of groups of equal windows over all ranks; 0 means
 *                     the slices ARE the LMS suffixes in suffix order
 * Replaces, for a sharded text, src/table.rs:411-416 (LMS placement), :421-448
 * (first induce) and :450-482 (compaction + naming). */
typedef struct {
    uint64_t n_total;        /* bytes of the whole text                                 */
    uint64_t m_total;        /* LMS suffixes of the whole text                          */
    uint64_t m_local;        /* LMS suffixes of this shard                              */
    uint64_t lo;             /* global offset of this shard                             */
    uint64_t recv_count;     /* entries of this rank's slice of the global order        */
    uint64_t distinct_local; /* distinct windows in the slice                           */
    uint64_t name_offset;    /* distinct windows on lower ranks                         */
    uint64_t ties_total;     /* members of non-singleton window groups, all ranks       */
    double   bytes_sent;     /* payload this rank sent to OTHER ranks (NVLink)          */
    double   bytes_recv;
    uint32_t kc;             /* characters per window                                   */
    uint32_t nranks, rank;
    uint32_t reserved;
} b200sa_shard_stats;

int b200sa_comm_unique_id(uint8_t *id128_out);
int b200sa_comm_init(b200sa_ctx *ctx, int nranks, int rank, const uint8_t *id128);
int b200sa_comm_attach(b200sa_ctx *ctx, void *nccl_comm);
int b200sa_comm_destroy(b200sa_ctx *ctx);
int b200sa_shard_lms_sort(b200sa_ctx *ctx, const uint8_t *d_shard, uint64_t len,
                          unsigned long long *d_sorted_gpos, uint32_t *d_names, uint64_t cap,
                          b200sa_shard_stats *out, void *stream);

/* Sharded lcp_lens (collective; SURVEY.md 8e): d_text (n bytes), d_sa and d_lcp (n u32) are
 * device buffers on EVERY rank.  replicated == 0: rank 0 holds text and table, they are
 * broadcast first; != 0: every rank already holds them.  Every rank computes Phi / PLCP for
 * its own range of text positions, the ranges are all-gathered, every rank turns its range of
 * ranks into LCP values, the slices are all-gathered: on return every rank holds the whole
 * lcp array, equal to lcp_lens_quadratic(text, table) (src/table.rs:348-361).  Every rank
 * checks that the table is a permutation and that it is the suffix array; all ranks hold the
 * same table and reach the same verdict.  A permutation that is not the suffix array is not
 * sharded: every rank computes the whole array with the uncapped per-pair compare (see
 * b200sa_lcp) and no collective runs after the check. */
int b200sa_lcp_sharded(b200sa_ctx *ctx, uint8_t *d_text, uint64_t n, uint32_t *d_sa, uint32_t *d_lcp,
                       int replicated, void *stream);

/* ---- introspection (bench / tests) ---- */

typedef struct {
    uint64_t n;               /* text bytes of the last build                     */
    uint64_t m;               /* LMS suffixes at level 0                          */
    uint64_t names;           /* robust path: distinct LMS substrings (reduced alphabet);
                                 direct path: LMS suffixes settled by the first window */
    uint32_t doubling_rounds; /* robust path: rank-pair doubling rounds on the reduced
                                 string; direct path: window rounds of the LMS sort */
    uint32_t kernel_launches; /* kernels launched by the last call                */
    uint32_t induce_blocks;   /* grid of the persistent induce kernels            */
    uint32_t sm_count;
    uint64_t workspace_bytes; /* device workspace currently held                  */
    uint32_t direct_sort;     /* 1: LMS suffixes sorted directly by character windows;
                                 0: robust path (stage-1 induce + naming + doubling) */
    uint32_t reserved;
} b200sa_stats;

int b200sa_last_stats(b200sa_ctx *ctx, b200sa_stats *out);

/* Per-phase device times (CUDA events on the launching stream) of the last
 * call.  Enable with b200sa_set_timing(ctx, 1).  Returns the number of phases;
 * fills up to cap entries.  names[i] points to static strings. */
int b200sa_set_timing(b200sa_ctx *ctx, int enabled);
int b200sa_last_phase_times(b200sa_ctx *ctx, const char **names, float *ms, int cap);

const char *b200sa_strerror(int code);
const char *b200sa_last_error(b200sa_ctx *ctx);   /* detail of the last failure */
const char *b200sa_version(void);

#ifdef __cplusplus
}
#endif
#endif /* B200SA_H */

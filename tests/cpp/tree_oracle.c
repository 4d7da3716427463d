/* tree_oracle.c -- CPU oracle of the suffix tree (test infrastructure only).
 *
 * A C restatement of the reference's `to_suffix_tree` (suffix_tree/src/lib.rs:392-505):
 * suffixes are inserted serially in suffix-array order; each insertion climbs from the
 * last inserted leaf to the first ancestor whose path length is <= lcp[i], then either
 * hangs a new leaf below it or splits its rightmost edge with a new internal node.  The
 * root starts as a leaf of suffix n with an empty label (`SuffixTree::init`).
 *
 * Children are kept in first-byte order.  Every insertion adds the largest key of its
 * parent (suffixes arrive in lexicographic order), so a doubly linked child list with
 * append / remove-last is the reference's BTreeMap for the operations the algorithm uses;
 * the key order is asserted on every append, as the reference asserts absence.
 *
 * The tree is emitted in preorder (children by first byte, = the reference's preorder())
 * as structure-of-arrays: parent (0xFFFFFFFF for the root), string depth, rank interval
 * [lo, hi), end (one past the subtree), nchildren, terminal flag and the label's start
 * offset in the text (where the reference's insertion order left it). */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define NONE 0xFFFFFFFFu

typedef struct {
    uint32_t parent, first, last, next, prev;   /* child list in key order */
    uint32_t start, end, path_len;              /* label = text[start, end) */
    uint32_t rank;                              /* leaf: its rank in the table; else NONE */
    uint32_t nch;
} node_t;

static uint32_t label_len(const node_t *t) { return t->end - t->start; }

static void set_parent(node_t *T, uint32_t c, uint32_t p) {
    T[c].parent = p;
    T[c].path_len = T[p].path_len + label_len(&T[c]);
}

/* append c as the largest key of p; -1 if the key order would break */
static int append_child(node_t *T, const uint8_t *text, uint32_t p, uint32_t c) {
    uint32_t l = T[p].last;
    if (l != NONE && text[T[l].start] >= text[T[c].start]) return -1;
    T[c].prev = l;
    T[c].next = NONE;
    if (l == NONE) T[p].first = c; else T[l].next = c;
    T[p].last = c;
    T[p].nch++;
    return 0;
}

static uint32_t remove_last_child(node_t *T, uint32_t p) {
    uint32_t l = T[p].last;
    uint32_t pv = T[l].prev;
    T[p].last = pv;
    if (pv == NONE) T[p].first = NONE; else T[pv].next = NONE;
    T[p].nch--;
    return l;
}

static uint32_t new_node(node_t *T, uint32_t *count, uint32_t start, uint32_t end, uint32_t rank) {
    uint32_t k = (*count)++;
    node_t *t = &T[k];
    t->parent = t->first = t->last = t->next = t->prev = NONE;
    t->start = start; t->end = end; t->path_len = 0; t->rank = rank; t->nch = 0;
    return k;
}

/* Returns 0, -1 on a broken invariant of the reference's algorithm, -2 out of memory.
 * Output arrays hold max(2n, 1) entries; *num_nodes gets the node count. */
int oracle_suffix_tree(const uint8_t *text, uint64_t n, const uint32_t *sa, const uint32_t *lcp,
                       uint32_t *parent, uint32_t *depth, uint32_t *lo, uint32_t *hi, uint32_t *end,
                       uint32_t *nchildren, uint8_t *terminal, uint32_t *start, uint64_t *num_nodes) {
    uint64_t cap = n ? 2 * n : 1;
    node_t *T = (node_t *)malloc(cap * sizeof(node_t));
    uint32_t *stack = (uint32_t *)malloc(cap * sizeof(uint32_t));
    uint32_t *pid = (uint32_t *)malloc(cap * sizeof(uint32_t));
    uint32_t *order = (uint32_t *)malloc(cap * sizeof(uint32_t));
    int rc = 0;
    if (!T || !stack || !pid || !order) { rc = -2; goto out; }
    uint32_t count = 0;
    uint32_t root = new_node(T, &count, 0, 0, NONE);      /* SuffixTree::init: leaf(n, 0, 0) */
    uint32_t last = root;
    for (uint64_t i = 0; i < n; i++) {
        uint32_t suf = sa[i], l = lcp[i];
        uint32_t v = last;                                 /* ancestor_lcp_len */
        while (T[v].path_len > l && T[v].parent != NONE) v = T[v].parent;
        uint32_t dv = T[v].path_len;
        if (dv == l) {
            uint32_t leaf = new_node(T, &count, suf + l, (uint32_t)n, (uint32_t)i);
            set_parent(T, leaf, v);
            if (append_child(T, text, v, leaf)) { rc = -1; goto out; }
            last = leaf;
        } else if (dv < l) {
            if (T[v].last == NONE) { rc = -1; goto out; }
            uint32_t r = remove_last_child(T, v);
            uint32_t prev = sa[i - 1];
            uint32_t in = new_node(T, &count, prev + dv, prev + l, NONE);
            set_parent(T, in, v);
            uint32_t rlen = T[r].path_len;
            T[r].start = prev + l;
            T[r].end = prev + rlen;
            set_parent(T, r, in);
            uint32_t leaf = new_node(T, &count, suf + l, (uint32_t)n, (uint32_t)i);
            set_parent(T, leaf, in);
            if (append_child(T, text, in, r) || append_child(T, text, in, leaf) || append_child(T, text, v, in)) {
                rc = -1;
                goto out;
            }
            last = leaf;
        } else {
            rc = -1;
            goto out;
        }
    }
    /* preorder: children by first byte */
    uint32_t sp = 0, k = 0;
    stack[sp++] = root;
    while (sp) {
        uint32_t u = stack[--sp];
        pid[u] = k;
        order[k++] = u;
        for (uint32_t c = T[u].last; c != NONE; c = T[c].prev) stack[sp++] = c;
    }
    for (uint32_t id = 0; id < count; id++) {
        const node_t *t = &T[order[id]];
        parent[id] = t->parent == NONE ? NONE : pid[t->parent];
        depth[id] = t->path_len;
        nchildren[id] = t->nch;
        terminal[id] = (t->rank != NONE || t->parent == NONE);
        start[id] = t->start;
        lo[id] = t->rank != NONE ? t->rank : NONE;
        hi[id] = t->rank != NONE ? t->rank + 1 : 0;
        end[id] = 1;                                       /* subtree size for now */
    }
    lo[0] = 0;
    hi[0] = (uint32_t)n;
    for (uint32_t id = count; id-- > 1;) {                 /* children before parents */
        uint32_t p = parent[id];
        if (lo[id] < lo[p]) lo[p] = lo[id];
        if (hi[id] > hi[p]) hi[p] = hi[id];
        end[p] += end[id];
    }
    for (uint32_t id = 0; id < count; id++) end[id] += id;
    *num_nodes = count;
out:
    free(T);
    free(stack);
    free(pid);
    free(order);
    return rc;
}

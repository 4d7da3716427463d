"""Suffix tree references for the tests (test infrastructure only).

* `oracle_tree(text)`: the C restatement of the reference's serial insertion
  (tests/cpp/tree_oracle.c), compiled on first use into a per-user temporary
  directory, so the repository tree is never written.
* `model_tree(text, sa, lcp)`: a numpy model of the data-parallel construction
  that libb200sa's `b200sa_suffix_tree_dev` runs (suffix_b200/csrc/tree.cuh):
  LCP intervals from all-nearest-smaller values, heads, absorbed intervals,
  preorder ids from a stable sort of the heads by left rank, O(1) parents.

Both return a dict of numpy arrays indexed by preorder id: parent (0xFFFFFFFF
for the root), depth (string depth), lo, hi (rank interval), end (one past the
subtree), nchildren; the oracle adds terminal and start (label offset).
"""
import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle import oracle

NONE = 0xFFFFFFFF
_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "cpp", "tree_oracle.c")
_lib = None


def _build() -> str:
    with open(_SRC, "rb") as f:
        tag = hashlib.sha256(f.read()).hexdigest()[:16]
    d = os.path.join(tempfile.gettempdir(), "b200sa-tree-oracle-%d" % os.getuid())
    os.makedirs(d, exist_ok=True)
    so = os.path.join(d, "libtree_oracle_%s.so" % tag)
    if not os.path.exists(so):
        tmp = so + ".%d.tmp" % os.getpid()
        subprocess.check_call(["gcc", "-O2", "-std=c11", "-Wall", "-Wextra", "-fPIC", "-shared",
                               "-o", tmp, _SRC])
        os.replace(tmp, so)
    return so


def lib():
    global _lib
    if _lib is None:
        L = ctypes.CDLL(_build())
        vp = ctypes.c_void_p
        L.oracle_suffix_tree.argtypes = [vp, ctypes.c_uint64, vp, vp] + [vp] * 8 + [ctypes.POINTER(ctypes.c_uint64)]
        L.oracle_suffix_tree.restype = ctypes.c_int
        _lib = L
    return _lib


def _u8(text) -> np.ndarray:
    if isinstance(text, str):
        text = text.encode("utf-8")
    return np.frombuffer(bytes(text), dtype=np.uint8)


def sa_lcp(text):
    t = _u8(text)
    sa = oracle.sais(t)
    return sa, oracle.lcp_kasai(t, sa)


FIELDS = ("parent", "depth", "lo", "hi", "end", "nchildren")


def oracle_tree(text, sa=None, lcp=None) -> dict:
    t = _u8(text)
    n = len(t)
    if sa is None:
        sa, lcp = sa_lcp(t)
    sa = np.ascontiguousarray(sa, dtype=np.uint32)
    lcp = np.ascontiguousarray(lcp, dtype=np.uint32)
    cap = max(2 * n, 1)
    out = {f: np.zeros(cap, dtype=np.uint32) for f in FIELDS + ("start",)}
    out["terminal"] = np.zeros(cap, dtype=np.uint8)
    k = ctypes.c_uint64(0)
    args = [out[f].ctypes.data for f in ("parent", "depth", "lo", "hi", "end", "nchildren", "terminal", "start")]
    rc = lib().oracle_suffix_tree(t.ctypes.data, n, sa.ctypes.data, lcp.ctypes.data, *args, ctypes.byref(k))
    assert rc == 0, "oracle_suffix_tree: %d" % rc
    return {f: a[:k.value].copy() for f, a in out.items()}


def oracle_labels(text, tree) -> list:
    """The reference's label bytes per preorder node: text[start, start + len)."""
    t = bytes(_u8(text))
    d, p, s = tree["depth"], tree["parent"], tree["start"]
    return [b""] + [t[int(s[u]):int(s[u]) + int(d[u] - d[p[u]])] for u in range(1, len(d))]


# ------------------------------------------------------------------ numpy model of tree.cuh
def ansv(lcp, strict=True):
    """Previous (left) and next (right) smaller values: strict '<', or '<=' when not strict."""
    n = len(lcp)
    vals = [int(v) for v in lcp]
    left = np.full(n, NONE, dtype=np.int64)
    right = np.full(n, n, dtype=np.int64)
    for idx, out in ((range(n), left), (range(n - 1, -1, -1), right)):
        st = []
        for i in idx:
            v = vals[i]
            while st and (vals[st[-1]] >= v if strict else vals[st[-1]] > v):
                st.pop()
            if st:
                out[i] = st[-1]
            st.append(i)
    return left, right


def model_tree(text, sa, lcp) -> dict:
    n = len(sa)
    sa = np.asarray(sa, dtype=np.int64)
    lcp = np.asarray(lcp, dtype=np.int64)
    if n <= 1:
        return {"parent": np.array([NONE, 0][:n + 1], dtype=np.uint32),
                "depth": np.array([0, 1][:n + 1], dtype=np.uint32),
                "lo": np.zeros(n + 1, dtype=np.uint32), "hi": np.full(n + 1, n, dtype=np.uint32),
                "end": np.full(n + 1, n + 1, dtype=np.uint32),
                "nchildren": np.array([n, 0][:n + 1], dtype=np.uint32)}
    psv, nsv = ansv(lcp, strict=True)
    pse, _ = ansv(lcp, strict=False)
    j = np.arange(n)
    suflen = n - sa                                   # string depth of leaf i
    boundary = (j >= 1) & (lcp > 0)
    head = boundary & (pse == psv)
    absorbed = np.zeros(n, dtype=bool)                # head j absorbed by leaf j-1
    absorbed[1:] = head[1:] & (lcp[1:] == suflen[:-1])
    keep = head & ~absorbed
    # heads in descending j, stably sorted by left rank: id = 1 + left + position
    hj = j[keep][::-1]
    order = np.argsort(psv[hj], kind="stable")
    hj, hl = hj[order], psv[hj][order]
    m = len(hj)
    headid = np.full(n, NONE, dtype=np.int64)
    headid[hj] = 1 + hl + np.arange(m)
    # base[l] = non-root nodes with left rank < l = l + heads with left < l
    e = np.zeros(n + 1, dtype=np.int64)
    last = np.ones(m, dtype=bool)
    last[:-1] = hl[1:] != hl[:-1]
    e[hl[last]] = np.arange(m)[last] + 1
    emax = np.maximum.accumulate(e)
    base = np.arange(n + 1) + np.concatenate(([0], emax[:-1]))
    cnt = 1 + n + m
    lcp_ext = np.concatenate((lcp, [0]))

    def head_of(b):
        while pse[b] != psv[b]:                      # <= 255 steps: children differ in first byte
            b = pse[b]
        return b

    def parent_of(l, r):
        b = l if lcp_ext[l] >= lcp_ext[r] else r
        if lcp_ext[b] == 0:
            return 0
        h = head_of(b)
        return base[psv[h] + 1] if absorbed[h] else headid[h]

    out = {f: np.zeros(cnt, dtype=np.int64) for f in FIELDS}
    out["parent"][0], out["hi"][0], out["end"][0] = NONE, n, cnt
    for i in range(n):
        u = base[i + 1]                               # leaf i: last node with left rank i
        absorbing = i + 1 < n and absorbed[i + 1]
        r = nsv[i + 1] if absorbing else i + 1
        out["lo"][u], out["hi"][u], out["depth"][u], out["end"][u] = i, r, suflen[i], 1 + base[r]
        out["parent"][u] = parent_of(i, r)
    for p in range(m):
        u, h = 1 + hl[p] + p, hj[p]
        out["lo"][u], out["hi"][u], out["depth"][u], out["end"][u] = psv[h], nsv[h], lcp[h], 1 + base[nsv[h]]
        out["parent"][u] = parent_of(psv[h], nsv[h])
    out["nchildren"] = np.bincount(out["parent"][1:], minlength=cnt)
    return {f: a.astype(np.uint32) for f, a in out.items()}

"""Suffix tree on the CPU: the C oracle (tests/cpp/tree_oracle.c) against a Python
restatement of the reference's insertion, the reference's KATs and quickcheck
properties, the numpy model of the device construction against the oracle, and
the C++ mirror (include/b200sa_tree.hpp) compiling."""
import os
import subprocess
import tempfile

import numpy as np
import pytest

from tests import tree_model as tm
from tests.families import adversarial

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

KAT_TEXTS = ["", "a", "aa", "banana", "apple", "mississippi", "☃abc☃", "zzzzabczzzzzabczzzzzz"]

# (label, terminals, #children, tree depth) in preorder
KAT_TREES = {
    "": [(b"", [0], 0, 0)],
    "a": [(b"", [1], 1, 0), (b"a", [0], 0, 1)],
    "aa": [(b"", [2], 1, 0), (b"a", [1], 1, 1), (b"a", [0], 0, 2)],
    "banana": [(b"", [6], 3, 0), (b"a", [5], 1, 1), (b"na", [3], 1, 2), (b"na", [1], 0, 3),
               (b"banana", [0], 0, 1), (b"na", [4], 1, 1), (b"na", [2], 0, 2)],
    "apple": [(b"", [5], 4, 0), (b"apple", [0], 0, 1), (b"e", [4], 0, 1), (b"le", [3], 0, 1),
              (b"p", [], 2, 1), (b"le", [2], 0, 2), (b"ple", [1], 0, 2)],
}


def restated_tree(text: bytes):
    """Direct restatement of to_suffix_tree (suffix_tree/src/lib.rs:392-505) with dict
    children; returns the preorder as (label, terminals, #children, tree depth)."""
    sa, lcp = tm.sa_lcp(text)
    n = len(text)

    def node(suf, start, end):
        return {"parent": None, "children": {}, "suffixes": [] if suf is None else [suf],
                "start": start, "end": end, "path_len": 0}

    def add_parent(c, p):
        c["parent"] = p
        c["path_len"] = p["path_len"] + c["end"] - c["start"]

    root = node(n, 0, 0)
    last = root
    for i, suf in enumerate(sa.tolist()):
        l = int(lcp[i])
        v = last
        while v["path_len"] > l and v["parent"] is not None:
            v = v["parent"]
        dv = v["path_len"]
        assert dv <= l
        leaf = node(suf, suf + l, n)
        if dv == l:
            add_parent(leaf, v)
            assert text[leaf["start"]] not in v["children"]
            v["children"][text[leaf["start"]]] = leaf
        else:
            r = v["children"].pop(max(v["children"]))
            prev = int(sa[i - 1])
            inner = node(None, prev + dv, prev + l)
            add_parent(inner, v)
            r["start"], r["end"] = prev + l, prev + r["path_len"]
            add_parent(r, inner)
            add_parent(leaf, inner)
            assert text[r["start"]] != text[leaf["start"]]
            inner["children"][text[r["start"]]] = r
            inner["children"][text[leaf["start"]]] = leaf
            v["children"][text[inner["start"]]] = inner
        last = leaf
    out, stack = [], [(root, 0)]
    while stack:
        u, d = stack.pop()
        out.append((text[u["start"]:u["end"]], u["suffixes"], len(u["children"]), d))
        stack.extend((u["children"][k], d + 1) for k in sorted(u["children"], reverse=True))
    return out


def oracle_preorder(text: bytes):
    o = tm.oracle_tree(text)
    labels = tm.oracle_labels(text, o)
    sa, _ = tm.sa_lcp(text)
    n = len(text)
    out = []
    for u in range(len(labels)):
        d, p = 0, o["parent"][u]
        while p != tm.NONE:
            d, p = d + 1, o["parent"][p]
        terms = [n] if u == 0 else ([int(sa[o["lo"][u]])] if o["terminal"][u] else [])
        out.append((labels[u], terms, int(o["nchildren"][u]), d))
    return out


def random_strings(count=500, seed=20260917):
    rng = np.random.default_rng(seed)
    alphabets = ["a", "ab", "abc", "acgt", None]
    out = []
    for k in range(count):
        n = int(rng.integers(0, 120))
        a = alphabets[k % len(alphabets)]
        if a is None:       # arbitrary code points, like quickcheck's String
            s = "".join(chr(int(c)) for c in rng.integers(1, 0x3000, n) if not 0xD800 <= c < 0xE000)
        else:
            s = "".join(a[int(c)] for c in rng.integers(0, len(a), n))
        out.append(s.encode("utf-8"))
    return out


@pytest.mark.parametrize("text", list(KAT_TREES))
def test_oracle_kat_values(text):
    assert oracle_preorder(text.encode()) == KAT_TREES[text]


@pytest.mark.parametrize("text", KAT_TEXTS)
def test_oracle_matches_restatement_kat(text):
    t = text.encode("utf-8")
    assert oracle_preorder(t) == restated_tree(t)


def test_oracle_matches_restatement_random():
    for t in random_strings(300, seed=7):
        assert oracle_preorder(t) == restated_tree(t), t


def check_properties(text: bytes, tree: dict, sa: np.ndarray):
    """The reference's quickcheck properties (suffix_tree/src/lib.rs:528-566), on node arrays."""
    n = len(text)
    lo, depth, nch, parent = tree["lo"], tree["depth"], tree["nchildren"], tree["parent"]
    ids = np.arange(len(parent))
    term = np.ones(len(parent), dtype=bool)                     # the root holds suffix n
    term[1:] = depth[1:].astype(np.int64) == n - sa[lo[1:]].astype(np.int64)
    length = np.zeros(len(parent), dtype=np.int64)
    length[1:] = depth[1:].astype(np.int64) - depth[parent[1:]]
    leaves = ids[term & (length > 0)]
    assert len(leaves) == n                                     # qc_n_leaves
    assert np.all(nch[~term] >= 2)                              # qc_internals_have_at_least_two_children
    assert np.array_equal(sa[lo[leaves]], sa)                   # qc_tree_enumerates_suffixes


def test_oracle_quickcheck_properties():
    for t in random_strings():
        sa, lcp = tm.sa_lcp(t)
        check_properties(t, tm.oracle_tree(t, sa, lcp), sa.astype(np.int64))


@pytest.mark.parametrize("name,text", adversarial(), ids=[a for a, _ in adversarial()])
def test_model_matches_oracle(name, text):
    sa, lcp = tm.sa_lcp(text)
    o, m = tm.oracle_tree(text, sa, lcp), tm.model_tree(text, sa, lcp)
    for f in tm.FIELDS:
        assert np.array_equal(o[f], m[f]), f


def test_model_matches_oracle_small():
    for t in random_strings(200, seed=11) + [k.encode("utf-8") for k in KAT_TEXTS]:
        sa, lcp = tm.sa_lcp(t)
        o, m = tm.oracle_tree(t, sa, lcp), tm.model_tree(t, sa, lcp)
        for f in tm.FIELDS:
            assert np.array_equal(o[f], m[f]), (t, f)


def build_cpp_tree_test() -> str:
    exe = os.path.join(tempfile.mkdtemp(prefix="b200sa-tree-cpp-"), "test_tree")
    src = os.path.join(ROOT, "tests", "cpp", "test_tree.cpp")
    lib = os.path.join(ROOT, "suffix_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-I", os.path.join(ROOT, "include"), src, "-o", exe,
                           "-L", lib, "-lb200sa", "-Wl,-rpath," + lib])
    return exe


def test_cpp_tree_mirror_compiles():
    assert os.path.exists(build_cpp_tree_test())

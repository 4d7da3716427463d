"""Suffix tree on the device (b200sa_suffix_tree / _dev, suffix_b200.SuffixTree): node arrays
entry for entry against the C restatement of the reference's insertion, both construction
paths, the reference's properties at 100 MB, the size limit and the C++ mirror."""
import ctypes
import subprocess

import numpy as np
import pytest

from suffix_b200 import B200SAError, SuffixTable, SuffixTree, _lib, gen
from tests import tree_model as tm
from tests.families import adversarial
from tests.test_tree import KAT_TEXTS, KAT_TREES, build_cpp_tree_test, check_properties

pytestmark = pytest.mark.gpu


def _check(text: bytes, tree: SuffixTree, labels: bool):
    sa, lcp = tm.sa_lcp(text)
    want = tm.oracle_tree(text, sa, lcp)
    a = tree.arrays()
    assert np.array_equal(a["sa"], sa)
    for f in tm.FIELDS:
        assert np.array_equal(a[f], want[f]), f
    if labels:                                  # leaf labels sum to O(n^2): small texts only
        got = [tree.label(u) for u in tree.root().preorder()]
        assert got == tm.oracle_labels(text, want)


def _both(text: bytes, labels: bool):
    _check(text, SuffixTree(text), labels)
    _check(text, SuffixTree.from_suffix_table(SuffixTable(text)), labels)


@pytest.mark.parametrize("text", KAT_TEXTS)
def test_tree_kat_arrays(text):
    _both(text.encode("utf-8"), labels=True)


@pytest.mark.parametrize("text", list(KAT_TREES))
def test_tree_kat_nodes(text):
    t = SuffixTree(text)
    got = [(t.label(u), u.suffixes(), len(u.children()), u.depth()) for u in t.root().preorder()]
    assert got == KAT_TREES[text]


def test_tree_node_api_banana():
    t = SuffixTree("banana")
    root = t.root()
    kids = list(root.children())
    assert [t.label(c) for c in kids] == [b"a", b"banana", b"na"]
    assert [t.label(c) for c in reversed(root.children())] == [b"na", b"banana", b"a"]
    deep = list(kids[0].preorder())[-1]
    assert [u.id for u in deep.ancestors()] == [3, 2, 1, 0]
    assert [u.suffixes() for u in root.leaves()] == [[5], [3], [1], [0], [4], [2]]
    assert root.suffix_indices().tolist() == [5, 3, 1, 0, 4, 2]
    assert kids[0].suffix_indices().tolist() == [5, 3, 1]
    assert root.has_terminals() and root.suffixes() == [6] and root.len() == 0
    assert t.text() == b"banana" and len(t) == 7


@pytest.mark.parametrize("name,text", adversarial(), ids=[a for a, _ in adversarial()])
def test_tree_adversarial(name, text):
    _both(text, labels=len(text) <= 3000)


@pytest.mark.parametrize("maker", ["dna", "english", "rand_bytes"])
def test_tree_1mb(maker):
    _both(getattr(gen, maker)(1_000_000).tobytes(), labels=False)


def test_tree_fixture_100k():
    _both(gen.fixture("AP009048_100000.fasta").tobytes(), labels=False)


def test_tree_dev_matches_host():
    """b200sa_suffix_tree_dev from SA + LCP in HBM, on the caller's stream."""
    import torch
    text = gen.english(1_000_000).tobytes()
    n = len(text)
    dev = torch.device("cuda:0")
    d_text = torch.frombuffer(bytearray(text), dtype=torch.uint8).to(dev)
    d_sa = torch.empty(n, dtype=torch.int32, device=dev)
    d_lcp = torch.empty(n, dtype=torch.int32, device=dev)
    ctx = _lib.Context(0)
    stream = torch.cuda.Stream(device=dev)
    ctx.build_lcp_dev(d_text.data_ptr(), n, d_sa.data_ptr(), d_lcp.data_ptr())
    torch.cuda.synchronize()                    # the context's stream -> the caller's stream
    out = {f: torch.full((2 * n,), 7, dtype=torch.int32, device=dev) for f in _lib.TREE_FIELDS}
    ctx.set_timing(True)
    k = ctx.suffix_tree_dev(d_text.data_ptr(), n, d_sa.data_ptr(), d_lcp.data_ptr(),
                            {f: t.data_ptr() for f, t in out.items()}, stream.cuda_stream)
    stream.synchronize()
    phases = dict(ctx.phase_times())
    assert {"tree_ansv", "tree_heads", "tree_sort", "tree_base", "tree_nodes"} <= set(phases)
    assert ctx.stats()["kernel_launches"] > 0
    host = SuffixTree(text)
    assert k == len(host)
    for f in _lib.TREE_FIELDS:
        assert np.array_equal(out[f][:k].cpu().numpy().view(np.uint32), host.arrays()[f]), f
    ctx.close()


@pytest.mark.parametrize("n", [0, 1])
def test_tree_dev_tiny_launches_nothing(n):
    import torch
    dev = torch.device("cuda:0")
    d_text = torch.zeros(max(n, 1), dtype=torch.uint8, device=dev)
    d_sa = torch.zeros(max(n, 1), dtype=torch.int32, device=dev)
    out = {f: torch.full((2,), 7, dtype=torch.int32, device=dev) for f in _lib.TREE_FIELDS}
    ctx = _lib.Context(0)
    k = ctx.suffix_tree_dev(d_text.data_ptr(), n, d_sa.data_ptr(), d_sa.data_ptr(),
                            {f: t.data_ptr() for f, t in out.items()})
    assert k == n + 1 and ctx.stats()["kernel_launches"] == 0
    want = tm.oracle_tree(b"a" * n)
    for f in tm.FIELDS:
        assert out[f][:k].cpu().numpy().view(np.uint32).tolist() == want[f].tolist(), f
    ctx.close()


def test_tree_dna_100mb_properties():
    """The reference's three properties, vectorised, on 100 MB of DNA."""
    text = gen.dna(100_000_000).tobytes()
    t = SuffixTree(text)
    a = t.arrays()
    assert len(t) <= 2 * len(text)
    check_properties(text, a, a["sa"].astype(np.int64))


def test_tree_too_large_before_any_access():
    ctx = _lib.Context(0)
    k = ctypes.c_uint64(0)
    null = _lib.Tree()
    n = 1 << 31
    rc = _lib.lib().b200sa_suffix_tree_dev(ctx._h, None, n, None, None, ctypes.byref(null), ctypes.byref(k), None)
    assert rc == -2
    rc = _lib.lib().b200sa_suffix_tree(ctx._h, None, n, None, 0, ctypes.byref(null), ctypes.byref(k))
    assert rc == -2
    ctx.close()


def test_tree_from_bad_table_raises():
    st = SuffixTable.from_parts(b"abc", np.array([0, 0, 1], dtype=np.uint32))
    with pytest.raises(B200SAError):
        SuffixTree.from_suffix_table(st)


def test_cpp_tree_mirror_kats():
    out = subprocess.run([build_cpp_tree_test()], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "cpp tree mirror ok" in out.stdout, out.stdout + out.stderr

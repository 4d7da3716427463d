"""CPU checks of the LCP dispatch on caller tables (tables given to lcp_lens through from_parts or
load, not built by the library), with the scalar model of lcp_dev in tests/lcp_path_model.py.

lcp_lens is defined for any permutation as lcp_lens_quadratic (src/table.rs:348-361): the common
prefix of each adjacent pair, whatever order the pairs are in.  The direct per-pair kernel has that
meaning; the linear Phi / PLCP path (Kasai) only has it on the suffix array.  These tests pin down
why the sortedness check in front of the linear path exists and that the checked dispatch is exact.
"""
import itertools

import numpy as np
import pytest

from oracle import oracle
from tests import families
from tests import lcp_path_model as model

KAT = families.kat()


def _u8(b: bytes) -> np.ndarray:
    return np.frombuffer(b, dtype=np.uint8)


def _cases_true_sa():
    out = [("kat_" + c["text"], c["text"].encode("utf-8")) for c in KAT["kat"]]
    out += [(name, data) for name, data in families.adversarial()]
    out += [("a^%d" % k, b"a" * k) for k in (255, 256, 257, 258, 300, 511, 512, 513, 1000)]
    return out


@pytest.mark.parametrize("name,data", _cases_true_sa(), ids=lambda x: x if isinstance(x, str) else "")
@pytest.mark.parametrize("linear", [False, True], ids=["default", "linear"])
def test_model_dispatch_true_sa(name, data, linear):
    """On the suffix array every path gives lcp_lens_quadratic, checked or not."""
    t = _u8(data)
    sa = oracle.sais(t)
    want = oracle.lcp_quadratic(t, sa)
    got, path, oob = model.device_lcp(t, sa, linear=linear)
    assert path in ("direct", "phi")                 # a true table never takes the unsorted branch
    assert not oob
    assert np.array_equal(got, want), (name, path)
    fused, fpath, _ = model.device_lcp(t, sa, linear=linear, fused=True)
    assert fpath == path and np.array_equal(fused, want)


def test_model_runs_around_cap():
    """a^n: rank r pairs suffixes of lengths r and r+1, so its LCP and its room are both r.  A pair
    is capped iff it reached 256 chars AND had room for more: r = 256 is exact, r > 256 is capped."""
    for n in (256, 257, 258):
        t = _u8(b"a" * n)
        sa = oracle.sais(t)
        _, capped = model.lcp_direct(t, sa, model.DIRECT_CAP)
        assert capped == max(0, n - 1 - 256), n
        _, path, _ = model.device_lcp(t, sa)
        assert path == ("direct" if n <= 257 else "phi"), n


def _texts_for_kinds():
    rng = np.random.default_rng(5)
    return [
        ("a^2000", b"a" * 2000),
        ("a^300", b"a" * 300),
        ("period8", (b"ACGTTGCA" * 40 + b"G") * 6),
        ("dna_repeat", _planted_repeat(rng, 4000, 600)),
        ("fixture_3k", families.gen.fixture("AP009048_10000.fasta").tobytes()[:3000]),
        ("bytes", rng.integers(0, 256, 3000, dtype=np.uint8).tobytes()),
        ("ab", b"ab" * 700),
    ]


def _planted_repeat(rng, n, rep):
    t = rng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), n)
    t[n // 2:n // 2 + rep] = t[100:100 + rep]
    return t.tobytes()


def _other_text(data: bytes) -> bytes:
    """A different text of the same length (last byte changed, then rotated)."""
    b = bytearray(data)
    b[-1] = (b[-1] + 1) % 256
    return bytes(b[len(b) // 3:] + b[:len(b) // 3])


@pytest.mark.parametrize("name,data", _texts_for_kinds(), ids=lambda x: x if isinstance(x, str) else "")
@pytest.mark.parametrize("linear", [False, True], ids=["default", "linear"])
def test_model_dispatch_every_table_kind(name, data, linear):
    """The checked dispatch equals lcp_lens_quadratic on every kind of caller table."""
    t = _u8(data)
    sa = oracle.sais(t)
    other = oracle.sais(_u8(_other_text(data)))
    for kind, tab in model.table_kinds(t, sa, np.random.default_rng(len(t)), other_sa=other):
        want = oracle.lcp_quadratic(t, tab)
        got, path, oob = model.device_lcp(t, tab, linear=linear)
        assert not oob, (kind, path)
        assert np.array_equal(got, want), (kind, path)
        sorted_ = oracle.verify_sa(t, tab) == 0
        if path != "direct":            # the check ran: the unsorted branch iff the table is not the SA
            assert (path == "phi") == sorted_, kind
        if kind == "true_sa":
            assert sorted_ and path != "unsorted"


def test_unchecked_phi_wrong_on_swapped_table():
    """Regression case: a^2000, the suffix array with ranks 700 and 701 swapped.  It passes the
    permutation check and 1744 pairs reach the direct cap, so the call goes to the linear path.
    Kasai's carry h is wrong there: without the sortedness check Phi / PLCP returns wrong values and
    reads past the end of the text (u32 `limit` wraps).  With the check the dispatch is exact."""
    t = _u8(b"a" * 2000)
    sa = oracle.sais(t)
    tab = sa.copy()
    tab[[700, 701]] = tab[[701, 700]]
    want = oracle.lcp_quadratic(t, tab)
    assert oracle.verify_sa(t, tab) != 0
    assert int((want >= 256).sum()) == 1744
    _, capped = model.lcp_direct(t, tab, model.DIRECT_CAP)
    assert capped == 1743                      # one pair of exactly 256 chars has no room for more
    got, path, oob = model.device_lcp(t, tab, check=False)
    assert path == "phi"
    assert int((got != want).sum()) == 14
    assert len(oob) == 14 and all(max(a, b) >= len(t) for a, b in oob)
    got, path, oob = model.device_lcp(t, tab)
    assert path == "unsorted" and not oob and np.array_equal(got, want)


def test_unchecked_phi_random_permutation():
    t = _u8(b"a" * 2000)
    tab = np.random.default_rng(1).permutation(2000)
    want = oracle.lcp_quadratic(t, tab)
    got, path, oob = model.device_lcp(t, tab, check=False)
    assert path == "phi" and (got != want).any() and oob
    got, path, oob = model.device_lcp(t, tab)
    assert path == "unsorted" and np.array_equal(got, want) and not oob


def _agrees(t, tab):
    assert model.is_suffix_array(t, tab) == (oracle.verify_sa(t, tab) == 0), (bytes(t), list(tab))


def test_sorted_check_matches_verify_sa_random():
    rng = np.random.default_rng(3)
    for n in (2, 3, 5, 17, 64, 257, 1000):
        for alpha in (b"a", b"ab", b"ACGT", bytes(range(256))):
            t = rng.choice(_u8(alpha), n)
            sa = oracle.sais(t)
            _agrees(t, sa)
            assert model.is_suffix_array(t, sa)
            for _ in range(5):
                _agrees(t, rng.permutation(n))
            for r in rng.choice(n - 1, size=min(n - 1, 8), replace=False):      # single adjacent swaps
                s = sa.copy()
                s[[r, r + 1]] = s[[r + 1, r]]
                _agrees(t, s)
                assert not model.is_suffix_array(t, s)
            i, j = sorted(rng.choice(n, size=2, replace=False))                 # one long-distance swap
            s = sa.copy()
            s[[i, j]] = s[[j, i]]
            _agrees(t, s)


def test_sorted_check_exhaustive_tiny():
    """Every text of 1-3 bytes over {a, b}, every permutation: covers the a+1 == n and b+1 == n
    edges of the neighbour test."""
    seen_true = 0
    for n in (1, 2, 3):
        for chars in itertools.product(b"ab", repeat=n):
            t = _u8(bytes(chars))
            for perm in itertools.permutations(range(n)):
                tab = np.array(perm, dtype=np.uint32)
                _agrees(t, tab)
                seen_true += oracle.verify_sa(t, tab) == 0
    assert seen_true == 2 + 4 + 8          # exactly one suffix array per text

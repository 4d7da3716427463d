"""Caller tables on the device: lcp_lens, the suffix tree and positions on tables the library did
not build (from_parts, load, the device-pointer entry points).

lcp_lens is defined for any permutation of 0..n-1 as lcp_lens_quadratic (src/table.rs:348-361), so
the expected value is always oracle.lcp_quadratic(text, table), entry for entry.  The tables are
mostly permutations that are NOT the suffix array: they pass the permutation check and must not
reach the Phi / PLCP path, which is only valid on the sorted table (tests/test_caller_tables.py
shows on the CPU what it computes otherwise).  The texts are chosen so that every branch of lcp_dev
sees them: capped direct pairs, the small and the binned Phi (n >= 2^22), and an 8-bit text above
32 MiB that goes straight to the linear path.
"""
import numpy as np
import pytest
from hypothesis import HealthCheck, given, settings, strategies as st

from oracle import oracle
from suffix_b200 import B200SAError, SuffixTable, SuffixTree, _lib, gen
from tests import lcp_path_model as model
from tests.test_gpu_tree import _check as check_tree

pytestmark = pytest.mark.gpu

# Upper bound on the sum of the per-pair LCPs of one case: an unsorted table costs the device the
# reference's quadratic compare, so a case above it would be a long-running kernel, not a test.
QUAD_BUDGET = 1_000_000_000
MODES = {"default": {}, "linear": {"B200SA_LCP_LINEAR": "1"}, "phi_direct": {"B200SA_PHI_DIRECT": "1"}}
CONTROL = gen.fixture("AP009048_10000.fasta")


@pytest.fixture(scope="module")
def ctx():
    c = _lib.Context(0)
    c.set_timing(True)
    yield c
    c.close()


def _planted(n: int, rep: int = 1000) -> np.ndarray:
    """DNA with one planted repeat of `rep` bytes (pairs above the direct cap)."""
    t = gen.dna(n).copy()
    t[n // 2:n // 2 + rep] = t[1000:1000 + rep]
    return t


def _other(t: np.ndarray) -> np.ndarray:
    """A different text of the same length (last byte changed, then rotated)."""
    o = t.copy()
    o[-1] = (int(o[-1]) + 1) % 256
    return np.roll(o, len(o) // 3)


def _sa(ctx, t: np.ndarray) -> np.ndarray:
    if len(t) <= 200_000:
        return oracle.sais(t)
    sa = ctx.build(t)
    assert oracle.verify_sa(t, sa) == 0
    return sa


def _want(t, tab) -> np.ndarray:
    want = oracle.lcp_quadratic(t, tab)
    assert int(want.sum(dtype=np.uint64)) <= QUAD_BUDGET
    return want


def _is_sa(t, tab) -> bool:
    return oracle.verify_sa(t, tab) == 0


def _phases(ctx):
    return [name for name, _ in ctx.phase_times()]


def _check_branch(names, is_sa):
    """An unsorted table never reaches Phi / PLCP; a sorted one never takes the unsorted branch, and
    reaches Phi only after the check."""
    if is_sa:
        assert "lcp_unsorted" not in names, names
        if "lcp_phi" in names:
            assert "lcp_sorted" in names and names.index("lcp_sorted") < names.index("lcp_phi"), names
    else:
        assert "lcp_phi" not in names and "lcp_plcp" not in names, names
        if "lcp_sorted" in names:
            assert "lcp_unsorted" in names, names


def _control(ctx):
    """The context is still usable: a valid build_lcp matches the oracle."""
    sa, lcp = ctx.build_lcp(CONTROL)
    want = oracle.sais(CONTROL)
    assert np.array_equal(sa, want)
    assert np.array_equal(lcp, oracle.lcp_quadratic(CONTROL, want))


TEXTS = {
    "a^3000": lambda: np.full(3000, 97, dtype=np.uint8),
    "a^20000": lambda: np.full(20000, 97, dtype=np.uint8),
    "period8": lambda: np.frombuffer((b"ACGTTGCA" * 40 + b"G") * 6, dtype=np.uint8).copy(),
    "fixture_tiled_50k": lambda: gen.tiled(gen.fixture("AP009048_10000.fasta"), 50_000),
    "dna_5M_repeat": lambda: _planted(5_000_000),
    "dna_2^22-1": lambda: _planted((1 << 22) - 1),
    "dna_2^22": lambda: _planted(1 << 22),
    "bytes_40M": lambda: gen.rand_bytes(40_000_000),
}


@pytest.mark.parametrize("name", list(TEXTS))
def test_lcp_every_table_kind(ctx, name, monkeypatch):
    """ctx.lcp (b200sa_lcp) on every table kind, in every LCP mode, entry for entry."""
    t = TEXTS[name]()
    n = len(t)
    sa = _sa(ctx, t)
    other = _sa(ctx, _other(t))
    for kind, tab in model.table_kinds(t, sa, np.random.default_rng(n), other_sa=other):
        want = _want(t, tab)
        is_sa = kind == "true_sa" or _is_sa(t, tab)
        assert is_sa == (kind == "true_sa"), kind
        for mode, env in MODES.items():
            with monkeypatch.context() as mp:
                for k, v in env.items():
                    mp.setenv(k, v)
                got = ctx.lcp(t, tab)
            names = _phases(ctx)
            assert np.array_equal(got, want), (name, kind, mode, names)
            _check_branch(names, is_sa)
        if not is_sa:
            _control(ctx)


def test_phases_true_sa_direct(ctx):
    """A true SA on DNA finishes on the direct path: the check never runs."""
    t = gen.dna(1_000_000)
    sa = ctx.build(t)
    assert np.array_equal(ctx.lcp(t, sa), oracle.lcp_quadratic(t, sa))
    names = _phases(ctx)
    assert "lcp_direct" in names and "lcp_sorted" not in names and "lcp_phi" not in names, names


@pytest.mark.parametrize("name", ["a^3000", "dna_linear"])
def test_phases_true_sa_phi(ctx, name, monkeypatch):
    """A true SA that reaches the linear path runs the check and then Phi / PLCP."""
    if name == "dna_linear":
        monkeypatch.setenv("B200SA_LCP_LINEAR", "1")
        t = gen.dna(1_000_000)
    else:
        t = TEXTS[name]()
    sa = _sa(ctx, t)
    assert np.array_equal(ctx.lcp(t, sa), oracle.lcp_quadratic(t, sa))
    names = _phases(ctx)
    for p in ("lcp_sorted", "lcp_phi", "lcp_plcp"):
        assert p in names, names
    assert names.index("lcp_sorted") < names.index("lcp_phi") < names.index("lcp_plcp")
    assert "lcp_unsorted" not in names


def test_fused_build_lcp_skips_check(ctx):
    """build_lcp built its own table: no check, even on the linear path."""
    t = TEXTS["a^3000"]()
    sa, lcp = ctx.build_lcp(t)
    assert np.array_equal(lcp, oracle.lcp_quadratic(t, sa))
    names = _phases(ctx)
    assert "lcp_phi" in names and "lcp_sorted" not in names, names


ENTRY_TEXTS = ["a^3000", "period8", "fixture_tiled_50k", "dna_2^22"]


def _entry_tables(t, sa):
    rng = np.random.default_rng(7)
    swapped = sa.copy()
    r = len(sa) // 3
    swapped[[r, r + 1]] = swapped[[r + 1, r]]
    return [("true_sa", sa), ("swapped", swapped), ("random_perm", rng.permutation(len(sa)).astype(np.uint32))]


@pytest.mark.parametrize("name", ENTRY_TEXTS)
def test_lcp_dev_unaligned(ctx, name):
    """b200sa_lcp_dev with a text pointer that is not 16-byte aligned."""
    import torch
    t = TEXTS[name]()
    n = len(t)
    sa = _sa(ctx, t)
    buf = torch.zeros(n + 1, dtype=torch.uint8, device="cuda")
    buf[1:] = torch.from_numpy(t)
    for kind, tab in _entry_tables(t, sa):
        want = _want(t, tab)
        d_sa = torch.from_numpy(tab.astype(np.int64)).cuda().to(torch.int32)
        d_lcp = torch.empty(n, dtype=torch.int32, device="cuda")
        ctx.lcp_dev(buf.data_ptr() + 1, n, d_sa.data_ptr(), d_lcp.data_ptr(), torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        assert np.array_equal(d_lcp.cpu().numpy().view(np.uint32), want), (name, kind)
        _check_branch(_phases(ctx), kind == "true_sa")
    _control(ctx)


@pytest.mark.parametrize("name", ENTRY_TEXTS)
def test_lcp_sharded_world1(ctx, name):
    """b200sa_lcp_sharded always uses Phi / PLCP on a sorted table, so every unsorted table is
    caught by the check."""
    import torch
    t = TEXTS[name]()
    n = len(t)
    sa = _sa(ctx, t)
    d_t = torch.from_numpy(t.copy()).cuda()
    for kind, tab in _entry_tables(t, sa):
        want = _want(t, tab)
        d_sa = torch.from_numpy(tab.astype(np.int64)).cuda().to(torch.int32)
        d_lcp = torch.empty(n, dtype=torch.int32, device="cuda")
        ctx.lcp_sharded(d_t.data_ptr(), n, d_sa.data_ptr(), d_lcp.data_ptr(), False,
                        torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        assert np.array_equal(d_lcp.cpu().numpy().view(np.uint32), want), (name, kind)
        names = _phases(ctx)
        assert "lcp_sorted" in names
        assert ("lcp_unsorted" in names) == (kind != "true_sa"), names
        assert ("lcps_plcp" in names) == (kind == "true_sa"), names
    _control(ctx)


@pytest.mark.parametrize("name", ["a^3000", "period8", "fixture_tiled_50k"])
def test_from_parts_and_load(name, tmp_path):
    """SuffixTable.from_parts(...).lcp_lens() and a save / load round trip of a swapped table."""
    t = TEXTS[name]()
    sa = oracle.sais(t)
    for kind, tab in _entry_tables(t, sa):
        want = _want(t, tab)
        st = SuffixTable.from_parts(t.tobytes(), tab)
        assert np.array_equal(st.lcp_lens(), want), (name, kind)
        path = str(tmp_path / kind)
        st.save(path)
        for mmap in (True, False):
            back = SuffixTable.load(path, mmap=mmap)
            assert np.array_equal(np.asarray(back.table()), tab)
            assert np.array_equal(back.lcp_lens(), want), (name, kind, mmap)
    ok = SuffixTable(CONTROL.tobytes())
    assert np.array_equal(ok.lcp_lens(), oracle.lcp_quadratic(CONTROL, oracle.sais(CONTROL)))


def _tree_texts():
    return [b"banana", b"mississippi", b"ab", b"aab", b"abab" * 50, b"a" * 3000,
            (b"ACGTTGCA" * 40 + b"G") * 6, CONTROL.tobytes()[:5000]]


@pytest.mark.parametrize("text", _tree_texts(), ids=lambda b: "%r" % b[:12])
def test_tree_rejects_unsorted_table(text):
    """from_suffix_table on a permutation that is not the suffix array: B200SA_ERR_BAD_ARG (the
    reference's tree construction asserts on such tables); the true table still gives the tree."""
    t = np.frombuffer(text, dtype=np.uint8)
    sa = oracle.sais(t)
    rejected = 0
    for kind, tab in model.table_kinds(t, sa, np.random.default_rng(len(t))):
        if _is_sa(t, tab):
            continue
        with pytest.raises(B200SAError) as e:
            SuffixTree.from_suffix_table(SuffixTable.from_parts(text, tab))
        assert e.value.code == -1, kind
        assert "suffix array" in str(e.value)
        rejected += 1
    assert rejected >= 3
    check_tree(text, SuffixTree.from_suffix_table(SuffixTable.from_parts(text, sa)), labels=len(text) <= 600)


# ------------------------------------------------------------ positions on any permutation
def _positions_dev(text: bytes, tab, qs, lead: int = 0):
    """b200sa_positions_dev; `lead` bytes of padding in front of the query batch."""
    import torch
    ctx = _lib.default_context(0)
    n = len(text)
    flat = b"\x5a" * lead + b"".join(qs)
    off = (lead + np.cumsum([0] + [len(q) for q in qs])).astype(np.int64)
    dev = torch.device("cuda:0")
    d_t = torch.from_numpy(np.frombuffer(text, dtype=np.uint8).copy()).to(dev) if n else torch.zeros(1, dtype=torch.uint8, device=dev)
    d_sa = torch.from_numpy(np.asarray(tab, dtype=np.int64)).to(dev).to(torch.int32) if n else torch.zeros(1, dtype=torch.int32, device=dev)
    d_q = torch.from_numpy(np.frombuffer(flat, dtype=np.uint8).copy() if flat else np.zeros(1, np.uint8)).to(dev)
    d_off = torch.from_numpy(off).to(dev)
    nq = len(qs)
    d_s = torch.full((max(nq, 1),), -7, dtype=torch.int32, device=dev)
    d_e = torch.full((max(nq, 1),), -7, dtype=torch.int32, device=dev)
    ctx.positions_dev(d_t.data_ptr(), n, d_sa.data_ptr(), d_q.data_ptr(), d_off.data_ptr(), nq,
                      d_s.data_ptr(), d_e.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    s, e = d_s.cpu().numpy(), d_e.cpu().numpy()
    return [(int(s[k]), int(e[k])) for k in range(nq)], ctx.stats()["kernel_launches"], (s, e)


def _check_positions(text: bytes, tab, qs, lead: int = 0):
    got, _, _ = _positions_dev(text, tab, qs, lead)
    t = np.frombuffer(text, dtype=np.uint8)
    for k, q in enumerate(qs):
        assert got[k] == oracle.positions(t, tab, q), (k, q)


def _queries(text: bytes, rng, nq: int):
    qs = []
    for _ in range(nq):
        ln = int(rng.integers(0, 12))
        if rng.random() < 0.7 and len(text) > ln:
            s = int(rng.integers(0, len(text) - ln + 1))
            qs.append(text[s:s + ln])
        else:
            qs.append(bytes(rng.choice(np.frombuffer(b"ab\x00\xff", dtype=np.uint8), ln).tolist()))
    return qs


@pytest.mark.parametrize("text", [b"a" * 500, b"ab" * 300, b"abaababaab" * 40, b"mississippi", b"\x00\xff" * 100],
                         ids=lambda b: "%r" % b[:10])
def test_positions_random_permutation(text):
    """positions_dev restates the reference's two binary searches, so on ANY permutation it returns
    what the reference's search over that table returns."""
    rng = np.random.default_rng(len(text))
    qs = _queries(text, rng, 3000)
    for seed in range(4):
        tab = np.random.default_rng(seed).permutation(len(text)).astype(np.uint32)
        _check_positions(text, tab, qs)
    _check_positions(text, oracle.sais(np.frombuffer(text, dtype=np.uint8)), qs)


@settings(max_examples=60, deadline=None, suppress_health_check=list(HealthCheck))
@given(st.binary(max_size=200), st.integers(0, 2 ** 32 - 1), st.data())
def test_prop_positions_any_permutation(text, seed, data):
    tab = np.random.default_rng(seed).permutation(len(text)).astype(np.uint32)
    subs = st.integers(0, len(text)).flatmap(lambda i: st.integers(i, len(text)).map(lambda j: text[i:j]))
    qs = data.draw(st.lists(st.one_of(st.binary(max_size=6), subs), min_size=1, max_size=24))
    _check_positions(text, tab, qs)


def test_positions_edges():
    text = b"abracadabra\x00cadabra\xff"
    t = np.frombuffer(text, dtype=np.uint8)
    sa = oracle.sais(t)
    first, last = text[int(sa[0]):], text[int(sa[-1]):]
    qs = [b"", b"a", b"", text + b"a", text, last + b"\x00", last + b"\xff", first[:max(1, len(first) - 1)],
          b"\x00", b"\x00\x00", b"\xff", b"\xff\xff", b"abra", b"", b"cad", b"zzz", b"\x00cad"]
    for lead in (0, 1, 3):                          # queries at odd byte offsets of the batch
        _check_positions(text, sa, qs, lead)
        _check_positions(text, sa[::-1].copy(), qs, lead)
    # nq = 0: no kernel launch, outputs untouched
    got, launches, (s, e) = _positions_dev(text, sa, [])
    assert got == [] and launches == 0 and int(s[0]) == -7 and int(e[0]) == -7
    # n = 0 and n = 1 with queries
    got, _, _ = _positions_dev(b"", np.zeros(0, dtype=np.uint32), [b"a", b"", b"\x00"])
    assert got == [(0, 0)] * 3
    for one in (b"a", b"\x00", b"\xff"):
        qs1 = [one, b"", one * 2, b"b", b"\x00", b"\xff"]
        tab1 = np.zeros(1, dtype=np.uint32)
        _check_positions(one, tab1, qs1)
        got, _, _ = _positions_dev(one, tab1, qs1)
        assert got[0] == (0, 1) and got[1] == (0, 0) and got[2] == (0, 0)

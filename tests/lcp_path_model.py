"""Scalar restatement of the device LCP dispatch (lcp_dev in suffix_b200/csrc/b200sa.cu and the
kernels of pipeline_kernels.cuh), for checking its rules on the CPU:

  * k_lcp_direct: the reference's per-pair compare (src/table.rs:348-361) capped at 256 chars;
    a pair is counted as capped when it reached the cap and had room for more.  Any capped pair
    sends the call to the linear path.
  * k_sa_inverse + k_sa_sorted: the check that a caller table is THE suffix array (the neighbour
    test of oracle_verify_sa), run before the linear path on tables the library did not build.
    A permutation that fails it gets the per-pair compare with no cap.
  * k_phi + k_plcp_samples + k_plcp + k_lcp_gather: Kasai's algorithm as Phi / two-level PLCP,
    LCP_CHUNK = 32 positions per thread, 32 samples per group, the h - 32 and h - 1 carries and
    the u32 `limit` arithmetic.  Reads at or past the end of the text are recorded (and the compare
    stops there) instead of performed.

Values only: how the device splits a compare between one lane and the warp does not change them.
Pure Python + numpy, test infrastructure only.
"""
import numpy as np

M32 = (1 << 32) - 1
PHI_NONE = M32
LCP_CHUNK = 32
SAMPLE_GROUP = 32
DIRECT_CAP = 256
DIRECT_MAX_N_8BIT = 32 << 20          # an 8-bit text above this goes straight to the linear path


def _u8(text) -> np.ndarray:
    if isinstance(text, str):
        text = text.encode("utf-8")
    if isinstance(text, (bytes, bytearray, memoryview)):
        return np.frombuffer(bytes(text), dtype=np.uint8)
    return np.ascontiguousarray(text, dtype=np.uint8)


def _common(t: np.ndarray, a: int, b: int, limit: int) -> int:
    """Equal leading bytes of t[a..) and t[b..), at most `limit` (all indices in range)."""
    k, step = 0, 64
    while k < limit:
        s = min(step, limit - k)
        x, y = t[a + k:a + k + s], t[b + k:b + k + s]
        if np.array_equal(x, y):
            k += s
            step = min(step * 2, 1 << 16)
        else:
            return k + int(np.flatnonzero(x != y)[0])
    return k


def _match(t: np.ndarray, n: int, a: int, b: int, limit: int, oob: list) -> int:
    """text_match with a u32 `limit` that may have wrapped: compares up to `limit` chars, records
    the first read at or past n and stops there."""
    safe = max(0, min(limit, n - max(a, b)))
    k = _common(t, a, b, safe)
    if k < safe or k == limit:
        return k
    oob.append((a + k, b + k))
    return k


def bits_of(text) -> int:
    """Bits per char of the packed text: 2 for <= 4 distinct bytes, 4 for <= 16, else 8 (raw)."""
    sigma = len(np.unique(_u8(text)))
    return 2 if sigma <= 4 else 4 if sigma <= 16 else 8


def lcp_direct(text, sa, cap: int):
    """k_lcp_direct -> (lcp, number of capped pairs)."""
    t, sa = _u8(text), np.asarray(sa, dtype=np.int64)
    n = len(t)
    lcp = np.zeros(n, dtype=np.int64)
    capped = 0
    for r in range(1, n):
        a, b = int(sa[r - 1]), int(sa[r])
        room = n - max(a, b)
        h = _common(t, a, b, min(room, cap))
        lcp[r] = h
        if h == cap and room > cap:
            capped += 1
    return lcp, capped


def is_suffix_array(text, sa) -> bool:
    """k_sa_inverse + k_sa_sorted on a permutation of 0..n-1."""
    t, sa = _u8(text), np.asarray(sa, dtype=np.int64)
    n = len(t)
    if n < 2:
        return True
    inv = np.empty(n, dtype=np.int64)
    inv[sa] = np.arange(n)
    a, b = sa[:-1], sa[1:]
    ca, cb = t[a].astype(np.int64), t[b].astype(np.int64)
    na = np.minimum(a + 1, n - 1)
    nb = np.minimum(b + 1, n - 1)
    wrong = np.where(ca != cb, ca > cb,
                     np.where(a + 1 == n, False,
                              np.where(b + 1 == n, True, inv[na] >= inv[nb])))
    return not bool(wrong.any())


def lcp_phi(text, sa):
    """Phi / two-level PLCP with no check of the table -> (lcp, reads at or past n)."""
    t, sa = _u8(text), np.asarray(sa, dtype=np.int64)
    n = len(t)
    oob = []
    if n == 0:
        return np.zeros(0, dtype=np.int64), oob
    phi = np.empty(n, dtype=np.int64)
    phi[sa[0]] = PHI_NONE
    phi[sa[1:]] = sa[:-1]
    nchunk = (n + LCP_CHUNK - 1) // LCP_CHUNK
    samp = np.zeros(nchunk, dtype=np.int64)
    for g in range((nchunk + SAMPLE_GROUP - 1) // SAMPLE_GROUP):       # k_plcp_samples, one thread
        h = 0
        for j in range(SAMPLE_GROUP):
            s = g * SAMPLE_GROUP + j
            i = s * LCP_CHUNK
            if i >= n:
                continue
            jp = int(phi[i])
            if jp == PHI_NONE:
                h = 0
            else:
                a, b = (i + h) & M32, (jp + h) & M32
                h = (h + _match(t, n, a, b, (n - max(a, b)) & M32, oob)) & M32
            samp[s] = h
            h = h - LCP_CHUNK if h > LCP_CHUNK else 0
    plcp = np.zeros(n, dtype=np.int64)
    for c in range(nchunk):                                            # k_plcp, one thread
        i0 = c * LCP_CHUNK
        h = int(samp[c])
        plcp[i0] = h
        h = h - 1 if h else 0
        for i in range(i0 + 1, min(i0 + LCP_CHUNK, n)):
            j = int(phi[i])
            if j == PHI_NONE:
                plcp[i] = 0
                h = 0
                continue
            a, b = (i + h) & M32, (j + h) & M32
            h = (h + _match(t, n, a, b, (n - max(a, b)) & M32, oob)) & M32
            plcp[i] = h
            h = h - 1 if h else 0
    return plcp[sa], oob                                               # k_lcp_gather


def device_lcp(text, sa, *, linear: bool = False, fused: bool = False, check: bool = True):
    """lcp_dev's dispatch -> (lcp, path, reads at or past n); path is "direct", "unsorted" or "phi".
    linear: B200SA_LCP_LINEAR (no direct path).  fused: the table was built by the same call
    (build_lcp*), so it is not checked.  check=False restates the dispatch without the sortedness
    check (what lcp_dev did before it)."""
    t = _u8(text)
    n = len(t)
    if n == 0:
        return np.zeros(0, dtype=np.int64), "direct", []
    if not linear and (bits_of(t) < 8 or n <= DIRECT_MAX_N_8BIT):
        lcp, capped = lcp_direct(t, sa, DIRECT_CAP)
        if capped == 0:
            return lcp, "direct", []
    if check and not fused and not is_suffix_array(t, sa):
        return lcp_direct(t, sa, n)[0], "unsorted", []
    lcp, oob = lcp_phi(t, sa)
    return lcp, "phi", oob


def table_kinds(text, sa, rng, other_sa=None):
    """(name, table) pairs of caller tables for `text` with true suffix array `sa`: permutations
    that pass the permutation check, most of them not the suffix array.  other_sa: the suffix
    array of a different text of the same length (a mismatched save / load)."""
    sa = np.asarray(sa, dtype=np.uint32)
    n = len(sa)
    out = [("true_sa", sa.copy()), ("random_perm", rng.permutation(n).astype(np.uint32)),
           ("reversed", sa[::-1].copy()), ("identity", np.arange(n, dtype=np.uint32))]
    if n >= 2:
        t = sa.copy()
        for r in rng.choice(n - 1, size=min(5, n - 1), replace=False):
            t[[r, r + 1]] = t[[r + 1, r]]
        out.append(("adjacent_swaps", t))
        t = sa.copy()
        i, j = n // 5, n - 1 - n // 7
        t[[i, j]] = t[[j, i]]
        out.append(("long_swap", t))
        t = sa.copy()
        lo, hi = n // 3, n // 3 + max(2, n // 10)
        t[lo:hi] = np.roll(t[lo:hi], 1)
        out.append(("rotated_block", t))
    if other_sa is not None:
        out.append(("other_text_sa", np.asarray(other_sa, dtype=np.uint32).copy()))
    return out

"""ctypes loader for libb200sa.so.  There is no CPU fallback: if the CUDA
library is missing or no device is usable, every call raises."""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B200SA_LIB") or os.path.join(_HERE, "libb200sa.so")


class B200SAError(RuntimeError):
    def __init__(self, code, detail=""):
        self.code = code
        super().__init__("b200sa error %d (%s)%s" % (code, strerror(code), (": " + detail) if detail else ""))


class Stats(ctypes.Structure):
    _fields_ = [("n", ctypes.c_uint64), ("m", ctypes.c_uint64), ("names", ctypes.c_uint64),
                ("doubling_rounds", ctypes.c_uint32), ("kernel_launches", ctypes.c_uint32),
                ("induce_blocks", ctypes.c_uint32), ("sm_count", ctypes.c_uint32),
                ("workspace_bytes", ctypes.c_uint64), ("direct_sort", ctypes.c_uint32), ("reserved", ctypes.c_uint32)]


class ShardStats(ctypes.Structure):
    _fields_ = [("n_total", ctypes.c_uint64), ("m_total", ctypes.c_uint64), ("m_local", ctypes.c_uint64),
                ("lo", ctypes.c_uint64), ("recv_count", ctypes.c_uint64), ("distinct_local", ctypes.c_uint64),
                ("name_offset", ctypes.c_uint64), ("ties_total", ctypes.c_uint64),
                ("bytes_sent", ctypes.c_double), ("bytes_recv", ctypes.c_double),
                ("kc", ctypes.c_uint32), ("nranks", ctypes.c_uint32), ("rank", ctypes.c_uint32), ("reserved", ctypes.c_uint32)]


class Tree(ctypes.Structure):
    """b200sa_tree: the six node arrays (host or device pointers)."""
    _fields_ = [(f, ctypes.c_void_p) for f in ("parent", "depth", "lo", "hi", "end", "nchildren")]


TREE_FIELDS = tuple(f for f, _ in Tree._fields_)
TREE_MAX_N = 0x7FFFFFFF   # B200SA_TREE_MAX_N


_lib = None


def lib():
    """Loads libb200sa.so (built by __graft_entry__.build()); raises if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError("libb200sa.so is not built (run `python __graft_entry__.py`); "
                           "suffix_b200 has no CPU fallback")
    L = ctypes.CDLL(LIB_PATH)
    vp, u64, u32, ci = ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint32, ctypes.c_int
    sig = {
        "b200sa_ctx_create": ([ci, ctypes.POINTER(vp)], ci),
        "b200sa_ctx_destroy": ([vp], None),
        "b200sa_build": ([vp, vp, u64, vp], ci),
        "b200sa_lcp": ([vp, vp, u64, vp, vp], ci),
        "b200sa_build_lcp": ([vp, vp, u64, vp, vp], ci),
        "b200sa_build_dev": ([vp, vp, u64, vp, vp], ci),
        "b200sa_lcp_dev": ([vp, vp, u64, vp, vp, vp], ci),
        "b200sa_build_lcp_dev": ([vp, vp, u64, vp, vp, vp], ci),
        "b200sa_positions_dev": ([vp, vp, u64, vp, vp, vp, u32, vp, vp, vp], ci),
        "b200sa_shard_summary": ([vp, vp, u64, ci, ctypes.POINTER(ci), vp], ci),
        "b200sa_shard_classify": ([vp, vp, u64, ci, ci, ci, vp, vp, vp, u64, vp, ctypes.POINTER(u64), vp], ci),
        "b200sa_comm_unique_id": ([vp], ci),
        "b200sa_comm_init": ([vp, ci, ci, vp], ci),
        "b200sa_comm_attach": ([vp, vp], ci),
        "b200sa_comm_destroy": ([vp], ci),
        "b200sa_shard_lms_sort": ([vp, vp, u64, vp, vp, u64, ctypes.POINTER(ShardStats), vp], ci),
        "b200sa_doc_ids_dev": ([vp, vp, u64, vp, u32, vp, vp, vp], ci),
        "b200sa_lcp_intervals_dev": ([vp, vp, u64, vp, vp, vp], ci),
        "b200sa_lcp_sharded": ([vp, vp, u64, vp, vp, ci, vp], ci),
        "b200sa_suffix_tree_dev": ([vp, vp, u64, vp, vp, ctypes.POINTER(Tree), ctypes.POINTER(u64), vp], ci),
        "b200sa_suffix_tree": ([vp, vp, u64, vp, ci, ctypes.POINTER(Tree), ctypes.POINTER(u64)], ci),
        "b200sa_last_stats": ([vp, ctypes.POINTER(Stats)], ci),
        "b200sa_set_timing": ([vp, ci], ci),
        "b200sa_last_phase_times": ([vp, ctypes.POINTER(ctypes.c_char_p), ctypes.POINTER(ctypes.c_float), ci], ci),
        "b200sa_strerror": ([ci], ctypes.c_char_p),
        "b200sa_last_error": ([vp], ctypes.c_char_p),
        "b200sa_version": ([], ctypes.c_char_p),
        "b200sa_test_classify": ([vp, vp, u64, vp, vp, vp, vp, u64, ctypes.POINTER(u64)], ci),
        "b200sa_test_classify_fused": ([vp, vp, u64, vp, vp, vp, vp, u64, ctypes.POINTER(u64)], ci),
        "b200sa_test_scan": ([vp, vp, u64, ci, vp, ctypes.POINTER(u32)], ci),
        "b200sa_test_sort_pairs32": ([vp, vp, vp, u64, ci], ci),
        "b200sa_test_sort_pairs64": ([vp, vp, vp, u64, ci], ci),
        "b200sa_test_reduced_sa": ([vp, vp, u64, u32, vp, ctypes.POINTER(u32)], ci),
        "b200sa_debug_fetch": ([vp, ci, vp, u64], ctypes.c_int64),
    }
    for name, (args, res) in sig.items():
        fn = getattr(L, name)
        fn.argtypes = args
        fn.restype = res
    _lib = L
    return L


def strerror(code):
    try:
        return lib().b200sa_strerror(code).decode()
    except Exception:
        return "?"


class Context:
    """One CUDA device + stream + reusable device workspace (b200sa_ctx)."""

    def __init__(self, device: int = 0):
        self._h = ctypes.c_void_p()
        rc = lib().b200sa_ctx_create(device, ctypes.byref(self._h))
        if rc != 0:
            raise B200SAError(rc, "b200sa_ctx_create(device=%d)" % device)
        self.device = device

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            lib().b200sa_ctx_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise B200SAError(rc, lib().b200sa_last_error(self._h).decode())

    # ---- host-buffer API
    def build(self, text: np.ndarray) -> np.ndarray:
        sa = np.empty(len(text), dtype=np.uint32)
        self._check(lib().b200sa_build(self._h, text.ctypes.data, len(text), sa.ctypes.data))
        return sa

    def lcp(self, text: np.ndarray, sa: np.ndarray) -> np.ndarray:
        out = np.empty(len(text), dtype=np.uint32)
        self._check(lib().b200sa_lcp(self._h, text.ctypes.data, len(text), sa.ctypes.data, out.ctypes.data))
        return out

    def build_lcp(self, text: np.ndarray):
        sa = np.empty(len(text), dtype=np.uint32)
        lcp = np.empty(len(text), dtype=np.uint32)
        self._check(lib().b200sa_build_lcp(self._h, text.ctypes.data, len(text), sa.ctypes.data, lcp.ctypes.data))
        return sa, lcp

    # ---- device-pointer API (raw integer device pointers, e.g. torch .data_ptr())
    def build_dev(self, d_text: int, n: int, d_sa: int, stream: int = 0):
        self._check(lib().b200sa_build_dev(self._h, d_text, n, d_sa, stream))

    def lcp_dev(self, d_text: int, n: int, d_sa: int, d_lcp: int, stream: int = 0):
        self._check(lib().b200sa_lcp_dev(self._h, d_text, n, d_sa, d_lcp, stream))

    def build_lcp_dev(self, d_text: int, n: int, d_sa: int, d_lcp: int, stream: int = 0):
        self._check(lib().b200sa_build_lcp_dev(self._h, d_text, n, d_sa, d_lcp, stream))

    def positions_dev(self, d_text, n, d_sa, d_q, d_qoff, nq, d_start, d_end, stream: int = 0):
        self._check(lib().b200sa_positions_dev(self._h, d_text, n, d_sa, d_q, d_qoff, nq, d_start, d_end, stream))

    # ---- multi-GPU shards (SURVEY 8e)
    def shard_summary(self, d_shard: int, length: int, next_char: int, stream: int = 0) -> int:
        st = ctypes.c_int(0)
        self._check(lib().b200sa_shard_summary(self._h, d_shard, length, next_char, ctypes.byref(st), stream))
        return int(st.value)

    def shard_classify(self, d_shard: int, length: int, prev_char: int, next_char: int, tail_carry: int,
                       d_stype: int = 0, d_lms: int = 0, d_lmspos: int = 0, cap_lms: int = 0, stream: int = 0):
        hist = np.zeros(768, dtype=np.uint64)
        m = ctypes.c_uint64(0)
        self._check(lib().b200sa_shard_classify(self._h, d_shard, length, prev_char, next_char, tail_carry,
                                                d_stype, d_lms, d_lmspos, cap_lms, hist.ctypes.data,
                                                ctypes.byref(m), stream))
        return hist, int(m.value)

    # communicator of the sharded entry points: NCCL inside the library (resolved at run time)
    @staticmethod
    def comm_unique_id() -> bytes:
        buf = (ctypes.c_uint8 * 128)()
        rc = lib().b200sa_comm_unique_id(buf)
        if rc != 0:
            raise B200SAError(rc, "b200sa_comm_unique_id")
        return bytes(buf)

    def comm_init(self, nranks: int, rank: int, unique_id: bytes):
        buf = (ctypes.c_uint8 * 128).from_buffer_copy(unique_id)
        self._check(lib().b200sa_comm_init(self._h, nranks, rank, buf))

    def comm_destroy(self):
        self._check(lib().b200sa_comm_destroy(self._h))

    def shard_lms_sort(self, d_shard: int, length: int, d_gpos: int, d_names: int, cap: int, stream: int = 0) -> dict:
        """Collective (b200sa_shard_lms_sort): this rank's slice of the global LMS-suffix order."""
        st = ShardStats()
        self._check(lib().b200sa_shard_lms_sort(self._h, d_shard, length, d_gpos, d_names, cap, ctypes.byref(st), stream))
        return {f: getattr(st, f) for f, _ in ShardStats._fields_}

    def doc_ids_dev(self, d_pos: int, count: int, d_doc_starts: int, ndocs: int, d_doc: int, d_off: int, stream: int = 0):
        self._check(lib().b200sa_doc_ids_dev(self._h, d_pos, count, d_doc_starts, ndocs, d_doc, d_off, stream))

    def lcp_intervals_dev(self, d_lcp: int, n: int, d_psv: int, d_nsv: int, stream: int = 0):
        self._check(lib().b200sa_lcp_intervals_dev(self._h, d_lcp, n, d_psv, d_nsv, stream))

    def lcp_sharded(self, d_text: int, n: int, d_sa: int, d_lcp: int, replicated: bool = False, stream: int = 0):
        self._check(lib().b200sa_lcp_sharded(self._h, d_text, n, d_sa, d_lcp, 1 if replicated else 0, stream))

    def suffix_tree_dev(self, d_text: int, n: int, d_sa: int, d_lcp: int, d_out: dict, stream: int = 0) -> int:
        """b200sa_suffix_tree_dev: d_out maps each of TREE_FIELDS to a device pointer of
        max(2n, 1) u32; returns the node count."""
        k = ctypes.c_uint64(0)
        tree = Tree(*(d_out[f] for f in TREE_FIELDS))
        self._check(lib().b200sa_suffix_tree_dev(self._h, d_text, n, d_sa, d_lcp, ctypes.byref(tree),
                                                 ctypes.byref(k), stream))
        return int(k.value)

    def suffix_tree(self, text: np.ndarray, sa: np.ndarray = None):
        """b200sa_suffix_tree -> (sa, {field: u32 array of the node count}).  sa=None builds the
        table on the device (SuffixTree::new); a given table must be the suffix array of the
        text (from_suffix_table), anything else raises B200SAError."""
        n = len(text)
        cap = max(2 * n, 1)
        out = {f: np.empty(cap, dtype=np.uint32) for f in TREE_FIELDS}
        given = sa is not None
        sa = np.ascontiguousarray(sa, dtype=np.uint32) if given else np.empty(n, dtype=np.uint32)
        if len(sa) != n:
            raise ValueError("table length %d != text length %d" % (len(sa), n))
        k = ctypes.c_uint64(0)
        tree = Tree(*(out[f].ctypes.data for f in TREE_FIELDS))
        self._check(lib().b200sa_suffix_tree(self._h, text.ctypes.data, n, sa.ctypes.data, 1 if given else 0,
                                             ctypes.byref(tree), ctypes.byref(k)))
        return sa, {f: a[:k.value] for f, a in out.items()}

    # ---- introspection
    def set_timing(self, on: bool):
        self._check(lib().b200sa_set_timing(self._h, 1 if on else 0))

    def phase_times(self):
        names = (ctypes.c_char_p * 64)()
        ms = (ctypes.c_float * 64)()
        k = lib().b200sa_last_phase_times(self._h, names, ms, 64)
        return [(names[i].decode(), float(ms[i])) for i in range(max(0, min(k, 64)))]

    def stats(self) -> dict:
        s = Stats()
        self._check(lib().b200sa_last_stats(self._h, ctypes.byref(s)))
        return {f: int(getattr(s, f)) for f, _ in Stats._fields_}

    def debug_fetch(self, which: int, cap: int = 1 << 26) -> np.ndarray:
        out = np.empty(cap, dtype=np.uint32)
        k = lib().b200sa_debug_fetch(self._h, which, out.ctypes.data, cap)
        if k < 0:
            raise B200SAError(int(k))
        return out[:min(k, cap)].copy()


_default = {}


def default_context(device: int = 0) -> Context:
    """Lazily created per-device context used by SuffixTable."""
    if device not in _default:
        _default[device] = Context(device)
    return _default[device]

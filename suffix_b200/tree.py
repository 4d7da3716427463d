"""Host-side mirror of the reference's `SuffixTree` / `Node` (suffix_tree/src/lib.rs).

The tree is built on the GPU from SA + LCP (b200sa_suffix_tree, include/b200sa.h) and
kept as six u32 arrays indexed by preorder id (children in first-byte order, the
reference's `preorder()`): parent, depth (string depth), lo/hi (rank interval), end
(one past the subtree) and nchildren.  `Node` is a (tree, id) handle with the
reference's methods; labels and terminals follow from the table:

* label(u) = text[sa[lo] + depth(parent), sa[lo] + depth(u)),
* u has a terminal iff depth(u) == n - sa[lo(u)] (suffix sa[lo]); the root has
  suffix n and an empty label.  Like the reference, a leaf whose suffix is a
  prefix of the next suffix keeps its terminal and has children.
"""
import numpy as np

from . import _lib
from .table import SuffixTable, _as_bytes, _lock

NONE = 0xFFFFFFFF


class SuffixTree:
    """A suffix tree (suffix_tree/src/lib.rs:45-49)."""

    def __init__(self, text, device: int = 0, *, _table=None):
        """SuffixTree::new; with _table, SuffixTree::from_suffix_table.  Raises
        OverflowError above B200SA_TREE_MAX_N = 2^31-1 bytes (node ids are u32)."""
        self._text = _as_bytes(text)
        n = len(self._text)
        if n > _lib.TREE_MAX_N:
            raise OverflowError("text longer than 2^31-1 bytes (B200SA_TREE_MAX_N)")
        t = np.frombuffer(self._text, dtype=np.uint8)
        with _lock:                           # default context is not thread-safe
            ctx = _lib.default_context(device)
            self._sa, self._a = ctx.suffix_tree(t, _table)
        self._n = n

    @classmethod
    def from_suffix_table(cls, st: SuffixTable) -> "SuffixTree":
        """SuffixTree::from_suffix_table: the table is checked to be the suffix array of the
        text; any other table raises B200SAError (B200SA_ERR_BAD_ARG)."""
        return cls(st.text(), st._device, _table=np.asarray(st.table()))

    def text(self) -> bytes:
        return self._text

    def root(self) -> "Node":
        return Node(self, 0)

    def label(self, node: "Node") -> bytes:
        """The path label *into* `node` (empty for the root)."""
        u = node.id
        if u == 0:
            return b""
        s = int(self._sa[self._a["lo"][u]])
        return self._text[s + int(self._a["depth"][self._a["parent"][u]]):s + int(self._a["depth"][u])]

    def arrays(self) -> dict:
        """Node arrays by preorder id (parent, depth, lo, hi, end, nchildren) and the table ("sa")."""
        return dict(self._a, sa=self._sa)

    def __len__(self) -> int:
        return len(self._a["parent"])


class Children:
    """Children of a node in first-byte order; len()-able like the reference's ExactSizeIterator."""

    def __init__(self, tree: SuffixTree, u: int):
        self._tree, self._u = tree, u

    def __len__(self) -> int:
        return int(self._tree._a["nchildren"][self._u])

    def __iter__(self):
        end = self._tree._a["end"]
        stop = int(end[self._u])
        c = self._u + 1
        while c < stop:
            yield Node(self._tree, c)
            c = int(end[c])

    def __reversed__(self):
        return reversed(list(self))


class Node:
    """A node of a SuffixTree: a (tree, preorder id) handle (suffix_tree/src/lib.rs:52-59)."""
    __slots__ = ("tree", "id")

    def __init__(self, tree: SuffixTree, u: int):
        self.tree = tree
        self.id = int(u)

    def __eq__(self, other):
        return isinstance(other, Node) and other.tree is self.tree and other.id == self.id

    def __hash__(self):
        return hash((id(self.tree), self.id))

    def __repr__(self):
        return "Node(id=%d, len=%d, children=%d, terminals=%d)" % (
            self.id, self.len(), len(self.children()), len(self.suffixes()))

    def children(self) -> Children:
        return Children(self.tree, self.id)

    def parent(self):
        p = int(self.tree._a["parent"][self.id])
        return None if p == NONE else Node(self.tree, p)

    def ancestors(self):
        """This node, its parent, ..., the root."""
        u = self
        while u is not None:
            yield u
            u = u.parent()

    def preorder(self):
        """This node and its subtree in lexicographic order (ids id .. end-1)."""
        for u in range(self.id, int(self.tree._a["end"][self.id])):
            yield Node(self.tree, u)

    def leaves(self):
        """Nodes below (and including) this one with terminals and a non-empty label."""
        return (u for u in self.preorder() if u.len() > 0 and u.has_terminals())

    def suffix_indices(self) -> np.ndarray:
        """Suffix indices of the leaves below this node, in suffix order: table[lo:hi]."""
        a = self.tree._a
        return self.tree._sa[int(a["lo"][self.id]):int(a["hi"][self.id])]

    def len(self) -> int:
        """The size of the path label into this node."""
        a = self.tree._a
        if self.id == 0:
            return 0
        return int(a["depth"][self.id]) - int(a["depth"][a["parent"][self.id]])

    def depth(self) -> int:
        """Number of ancestors, not including self."""
        return sum(1 for _ in self.ancestors()) - 1

    def has_terminals(self) -> bool:
        return len(self.suffixes()) > 0

    def suffixes(self) -> list:
        t = self.tree
        if self.id == 0:
            return [t._n]
        s = int(t._sa[t._a["lo"][self.id]])
        return [s] if int(t._a["depth"][self.id]) == t._n - s else []

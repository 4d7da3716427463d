"""suffix_b200 -- B200-native suffix array / LCP construction behind the
BurntSushi/suffix `SuffixTable` API (see DESIGN.md).  The compute path is
libb200sa.so (hand-written sm_100a CUDA behind the C-ABI of include/b200sa.h);
there is no CPU fallback."""
from ._lib import B200SAError, Context, default_context  # noqa: F401
from .table import SuffixTable  # noqa: F401
from .generalized import GeneralizedSuffixTable  # noqa: F401,E402
from .tree import Node, SuffixTree  # noqa: F401,E402

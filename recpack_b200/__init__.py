"""recpack_b200 -- B200-native drop-in for RecPack's item-similarity hot path.

``ItemKNN`` (fit / predict) and ``NDCGK`` / ``RecallK`` / ... keep the reference's contracts -- they subclass the
reference's own classes when ``recpack`` is importable (``_ref.py``) -- and run on hand-written sm_100a CUDA
kernels through the C ABI in include/rpk.h.  There is no CPU fallback: without ``recpack_b200/librpk.so`` and
a B200 every compute call raises."""
from .base import Algorithm, ItemSimilarityMatrixAlgorithm, TopKItemSimilarityMatrixAlgorithm  # noqa: F401
from .matrix import UnsupportedTypeError, to_csr_matrix  # noqa: F401
from .metrics import NDCGK, DCGK, RecallK, CalibratedRecallK, PrecisionK, ReciprocalRankK, HitK, CoverageK  # noqa: F401
from .ease import EASE  # noqa: F401
from .embedding import embedding_top_k  # noqa: F401
from .factorization import FactorizationAlgorithm  # noqa: F401
from .nearest_neighbour import ItemKNN, pearson_top_k, real_top_k  # noqa: F401
from .postprocessing import ExcludeItems, SelectItems  # noqa: F401
from .splitters import FractionInteractionSplitter  # noqa: F401
from .util import get_top_K_ranks, get_top_K_values  # noqa: F401

from . import factorization as _factorization  # noqa: E402
from . import time_aware as _time_aware  # noqa: E402

for _n in _time_aware.__all__:  # TARSItemKNN drop-ins: only when recpack (InteractionMatrix, decay functions) is importable
    globals()[_n] = getattr(_time_aware, _n)
for _n in _factorization.__all__:  # SVD / NMF drop-ins: only when recpack is importable
    globals()[_n] = getattr(_factorization, _n)

__version__ = "0.1.0"

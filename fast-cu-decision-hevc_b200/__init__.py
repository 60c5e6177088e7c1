"""cucudecide - B200 (sm_100a) CU-decision cost engine for the HM-based Fast-CU-Decision-HEVC encoder.

This Python package is a thin ctypes binding over the C ABI of ``libcucudecide.so``
(``include/cucudecide.h``).  The product is the shared library; Python is only used by the tests
and by ``bench.py``.  There is no CPU compute path: if the library is missing or no sm_100 GPU is
visible, the calls raise.

The directory name contains hyphens, so import it with::

    import importlib; cucd = importlib.import_module("fast-cu-decision-hevc_b200")
"""
from .sharding import FORK_PERIOD, shard_independent, shard_pictures  # noqa: F401
from .binding import (  # noqa: F401
    COST_NOT_INSIDE,
    COST_PRUNED,
    CucdError,
    Engine,
    LIB_PATH,
    NUM_MODES,
    PACKED_CTU_BYTES,
    PUS_PER_CTU,
    RmdQueue,
    SEARCH_FRAC,
    SEARCH_HADAMARD,
    SEARCH_RESULT,
    SEARCH_TZ_2NX2N,
    TU_INTRA_SLICE,
    TU_SIGN_HIDING,
    TZ_DESC,
    declared_symbols,
    load_library,
    tcm_fit,
    unpack_costs,
)

"""tgp_b200: B200 (sm_100a) kernels for tgp's Reduce + Connect hot path behind the SRC operator API."""
from . import functional, unbatched
from .connect import B200DenseConnect, B200SparseConnect, Connect, sparse_connect
from .lift import B200Lift
from .functional import sparse_connect_padded
from .graphed import GraphedStep
from .poolers import (acc_pool, diff_pool, dmon_pool, hosc_pool, mincut_pool, patch_pooler, sparse_pool,
                      sparse_pool_padded)
from .reduce import B200Reduce, Reduce
from .select import topk, topk_select
from .select_output import SelectOutput, cluster_to_s

__all__ = [
    "functional", "B200Reduce", "B200SparseConnect", "B200DenseConnect", "B200Lift", "Reduce", "Connect", "SelectOutput",
    "cluster_to_s", "topk", "topk_select", "sparse_connect", "mincut_pool", "diff_pool", "dmon_pool", "acc_pool",
    "hosc_pool", "sparse_pool", "patch_pooler", "sparse_connect_padded", "sparse_pool_padded", "GraphedStep", "unbatched",
]
__version__ = "0.1.0"

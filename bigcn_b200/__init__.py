"""bigcn_b200 -- B200-native (sm_100a) BiGCN hot path behind the reference's module API.

    from bigcn_b200 import BiGCN, Net, TDrumorGCN, BUrumorGCN, GCNConv, EBGCN

The CUDA library (bigcn_b200/libbigcn_b200.so, C-ABI in include/bigcn_b200.h) is the
product; importing this package without it raises, and no op has a CPU fallback.
"""
from ._lib import BigcnError, LIB_PATH, lib  # noqa: F401

lib()  # fail loudly at import time if the CUDA library has not been built

from .nn import GCNConv, TDrumorGCN, BUrumorGCN, BiGCN, Net  # noqa: E402,F401
from .ebgcn import EBGCN  # noqa: E402,F401  (its TDrumorGCN / BUrumorGCN live in bigcn_b200.ebgcn)
from .trainer import FusedTrainer  # noqa: E402,F401
from . import data, ops, torch_ops  # noqa: E402,F401  (torch_ops registers torch.ops.bigcn_b200.*)
from .ops import SparseX, host_dense_to_csr  # noqa: E402,F401
from .loader import DeviceForest  # noqa: E402,F401
from . import ingest  # noqa: E402,F401
from .ingest import forest_from_raw  # noqa: E402,F401
from .metrics import EvalCounts  # noqa: E402,F401
from .feeder import HostFeeder  # noqa: E402,F401
from .training import train_GCN  # noqa: E402,F401
from .checkpoint import EarlyStopping, EarlyStopping2class, make_checkpoint  # noqa: E402,F401

__all__ = ["GCNConv", "TDrumorGCN", "BUrumorGCN", "BiGCN", "Net", "EBGCN", "FusedTrainer", "BigcnError",
           "SparseX", "host_dense_to_csr", "DeviceForest", "forest_from_raw", "ingest", "EvalCounts", "HostFeeder", "train_GCN", "EarlyStopping", "EarlyStopping2class", "make_checkpoint", "data", "ops", "torch_ops"]

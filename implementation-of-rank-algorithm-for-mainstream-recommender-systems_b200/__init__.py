"""rank_b200 — the CTR hot path of reallinshengxiang/Implementation-of-Rank-Algorithm-for-
Mainstream-Recommender-Systems on B200 (sm_100a).

The reference's model classes keep their names, constructor/forward signatures and state_dict
keys; their embedding gathers, feature-interaction layers and the sparse embedding-gradient
reduction run in hand-written CUDA kernels behind the C ABI of `include/rank_b200.h`
(`librank_b200.so`, loaded with ctypes).  There is no CPU fallback: without the library, or with
tensors that are not on a CUDA device, every op raises.

The directory name contains hyphens, so import it through the `rank_b200` alias at the repo root
(or `importlib.import_module`).
"""
from . import _lib
from ._lib import RankB200Error, check_index_errors, library_path
from .vocab import VOCAB_FILE, WECHAT_VOCAB_LINES, table_heights, write_vocab_dir
from .sparse import GatherConcat, GradSource, OccurrencePlan, gather_concat
from .deepfm import DeepFM
from .fwfm import FwFM
from .dcn import DCNModel, cross_layer
from .deepcrossing import DeepCrossingModel, residual_unit
from .din import (DIN, Dice, din_attention, din_collate_fn, get_activation_unit_precision,
                  set_activation_unit_precision)
from .afm import AFM, create_feature_columns
from .sharded import RowShardedEmbedding, shard_bst_feedid_table
from .bst import BSTModel, BSTTransformer, leakyrelu, load_vocabulary
from .staging import PackedBatch
from .loader import EncodedWechat
from .device_data import BatchFeed, DeviceWechat
from .optim import Adam, RowwiseAdam
from .metrics import BinaryMetrics

__all__ = [
    "RankB200Error", "check_index_errors", "library_path",
    "VOCAB_FILE", "WECHAT_VOCAB_LINES", "table_heights", "write_vocab_dir",
    "GradSource", "OccurrencePlan", "gather_concat",
    "DeepFM", "FwFM", "DCNModel", "cross_layer", "DeepCrossingModel", "residual_unit", "DIN", "Dice", "din_attention", "din_collate_fn", "set_activation_unit_precision",
    "get_activation_unit_precision",
    "AFM", "create_feature_columns", "RowShardedEmbedding", "shard_bst_feedid_table", "BSTModel", "BSTTransformer", "leakyrelu", "load_vocabulary",
    "PackedBatch", "EncodedWechat", "DeviceWechat", "BatchFeed", "Adam", "RowwiseAdam", "BinaryMetrics",
]

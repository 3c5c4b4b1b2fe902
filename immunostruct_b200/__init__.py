"""immunostruct_b200 -- B200-native (sm_100a) implementation of ImmunoStruct's training / inference
hot path behind the reference's own plug-in API (``model_map``, ``Losses``, ``PairedContrastiveLoss``,
``collate`` / ``batch``).  See DESIGN.md and INTEGRATION.md."""
from .graph import Graph, GraphBatch, batch, collate, collate_amino_acid, graph  # noqa: F401
from .layers import EGNNConv, MultiHeadAttention, SelfAttention  # noqa: F401
from .loss import Losses  # noqa: F401
from .contrastive import PairedContrastiveLoss  # noqa: F401
from .mapping import model_map  # noqa: F401
from .functional import get_precision, set_precision  # noqa: F401
from .loader import DevicePrefetcher  # noqa: F401
from .packed import PackedGraphBatch, PackedGraphDataset, PackedSequence, pack_graph_batch, pack_sequence  # noqa: F401
from .optim import FusedAdam, FusedAdamW  # noqa: F401
from .augment import TrainAugment  # noqa: F401
from .graphed import CapturedStep  # noqa: F401
from . import attribution, augment, dataloading, nn, optim, ops, predictive  # noqa: F401
from .ops import use_custom_ops  # noqa: F401
from .functional import invalidate_caches  # noqa: F401

DGLGraph = Graph     # `import immunostruct_b200 as dgl` keeps data/utils.py's isinstance checks working

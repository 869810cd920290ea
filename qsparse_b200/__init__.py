"""qsparse_b200 — the quantize/prune hot path of mlzxy/qsparse on hand-written
sm_100a CUDA kernels, behind qsparse's own Python API (export list of
``qsparse/__init__.py``).  CUDA only: there is no CPU or PyTorch-eager fallback."""
# fmt: off
from .convert import convert
from .fuse import fuse_bn
from .fused import fuse_prune_quantize
from .quantize import quantize, DecimalQuantizer, ScalerQuantizer, AdaptiveQuantizer, PercentileQuantizer
from .quantize import BlockScaledQuantizer, export_block_scaled, dequantize_block_scaled
from .sparse import MagnitudePruningCallback, UniformPruningCallback, prune, devise_layerwise_pruning_schedule
from .sparse import WeightSetPruner
from .graphs import GraphedTrainStep
from .util import auto_name_prune_quantize_layers, calculate_mask_given_importance
from .util import get_option as get_qsparse_option
from .util import set_options as set_qsparse_options
from .util import preload_qsparse_state_dict
# fmt: on

__version__ = "2.0.1+b200.1"

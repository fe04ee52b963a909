"""movae_b200 -- B200-native (sm_100a) drop-in for MO-VAE's per-step hot path: multi-objective
gradient aggregation (Gramian -> small solve -> recombine -> .grad) and the VQ quantizer.

CUDA-only by design: importing works anywhere, but every op raises if the in-tree library
`mo-vae_b200/lib/libmovae_b200.so` is missing or the tensors are not on a CUDA device."""
from . import ops, parallel  # noqa: F401
from ._lib import LIB_PATH, lib  # noqa: F401
from .aggregation import (COMFORT, IMTLG, MGDA, Aggregator, AlignedMTL, AlignedMTLWeighting, DualProj,  # noqa: F401
                          GramianWeightedAggregator, IMTLGWeighting, Mean, MGDAWeighting, NUPGrad, PCGrad, PCGradWeighting,
                          PNUPGrad, StableMGDA, Sum, UPGrad, UPGradWeighting, Weighting, beta_schedule, make_aggregator)
from .autojac import backward, mtl_backward  # noqa: F401
from .extract import CodeExtractor  # noqa: F401
from .host import HostAggregationPlan, aggregate_host  # noqa: F401
from .optim import (SGD, Adam, AdamW, FlatParameters, FusedOptimizer, GraphedStep, RMSprop, make_optimizer)  # noqa: F401
from .quantizer import VectorQuantizer, code_indices, codebook_usage_count  # noqa: F401

__version__ = "0.1.0"

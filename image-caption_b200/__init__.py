"""image-caption_b200: B200-native (sm_100a) drop-in for the caption-generator hot path of
shao-chi/Image-Caption (core/models.py + core/TRANSFORMER/).

The directory name contains a hyphen, so import it through `icap_loader.load()` at the repo root
(registers the package as `image_caption_b200`), or put this directory on sys.path and import the
drop-in tree `core.TRANSFORMER.model` / `core.models` exactly like the reference's.
"""
from .engine import ModelConfig, CaptionEngine, param_layout, flat_offsets   # noqa: F401
from .transformer import Transformer, PolicyNetwork, GraphedTrainStep, GraphedDecode, DataParallel, GradBuckets                       # noqa: F401
from .engine import RegionBatch                                              # noqa: F401
from .feed import RegionCache, PrefetchLoader                                # noqa: F401
from .metrics import CaptionScorer, CaptionReward                           # noqa: F401
from . import _native                                                        # noqa: F401

__all__ = ["Transformer", "PolicyNetwork", "GraphedTrainStep", "GraphedDecode", "DataParallel", "GradBuckets", "RegionCache", "RegionBatch", "PrefetchLoader", "ModelConfig", "CaptionEngine", "param_layout", "flat_offsets", "CaptionScorer", "CaptionReward"]

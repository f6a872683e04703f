"""marigold_b200 — B200-native (sm_100a) implementation of Marigold's denoising hot path.

Public surface mirrors the reference package (marigold/__init__.py:30-41) for the path in scope:
pipelines + output dataclasses + ensembling, plus the Engine that stands in for unet/vae/scheduler.
Importing the package does not load the CUDA library; the first Engine()/ensemble call does, and
fails loudly if it is unavailable (no CPU fallback)."""
from .engine import Engine, EngineConfig  # noqa: F401
from .ensemble import ensemble_depth, ensemble_iid, ensemble_normals  # noqa: F401
from .evaluation import align_depth_least_square, evaluate_depth, evaluate_iid, evaluate_normals  # noqa: F401
from .iid import IIDEntry, MarigoldIIDOutput  # noqa: F401
from .pipeline import (  # noqa: F401
    MarigoldDepthOutput,
    MarigoldDepthPipeline,
    MarigoldIIDPipeline,
    MarigoldNormalsOutput,
    MarigoldNormalsPipeline,
    MarigoldPipeline,
)
from .schedulers import DDIMScheduler, LCMScheduler  # noqa: F401

__all__ = ["Engine", "EngineConfig", "MarigoldDepthPipeline", "MarigoldNormalsPipeline", "MarigoldPipeline",
           "MarigoldDepthOutput", "MarigoldNormalsOutput", "DDIMScheduler", "LCMScheduler", "ensemble_depth",
           "ensemble_normals", "ensemble_iid", "IIDEntry", "MarigoldIIDOutput", "MarigoldIIDPipeline"]

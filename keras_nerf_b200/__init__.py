"""keras_nerf_b200 -- B200-native (sm_100a) drop-in for keras_nerf's per-ray hot path.

Mirrors the reference package layout (`data.rays`, `data.utils`, `model.nerf.{utils,mlp,nerf}`) and
keeps its class/call signatures; all math runs in libknerf.so (hand-written CUDA) through a C ABI.
"""
from .data.image import ImageLoader  # noqa: F401
from .data.llff import LLFFDatasetLoader  # noqa: F401
from .data.loader import DatasetLoader  # noqa: F401
from .data.rays import RaysGenerator  # noqa: F401
from .data.utils import get_focal_from_fov, pose_spherical  # noqa: F401
from .model.nerf.callback import NeRFTrainMonitor  # noqa: F401
from .model.nerf.mlp import NeRFMLP  # noqa: F401
from .model.nerf.nerf import NeRF  # noqa: F401
from .model.nerf.utils import NeRFUtils  # noqa: F401

__all__ = ["ImageLoader", "DatasetLoader", "LLFFDatasetLoader", "NeRFTrainMonitor", "RaysGenerator", "get_focal_from_fov", "pose_spherical", "NeRFMLP", "NeRF", "NeRFUtils"]

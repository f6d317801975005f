"""B200-native (sm_100a) pillar LiDAR-encoder hot path of Advaith-Sajeev/LiDAR-Vision-VQA's src/lidar-encoder:
point -> pillar grouping, per-pillar feature net (augment + Linear + BN + ReLU + max) and the dense BEV scatter,
behind the reference's own module interface.  See DESIGN.md and include/pillars_b200.h."""
from ._native import NativeLibraryError  # noqa: F401
from .modules import (MAP_TO_BEV_REGISTRY, VFE_REGISTRY, DynamicPillarVFE, DynamicPillarVFESimple2D,  # noqa: F401
                      PFNLayer, PillarVFE, PillarVFEFromPoints, PointPillarScatter, PointPillarScatter3d, VFETemplate)
from .backbone import BaseBEVBackbone, BaseBEVResBackbone  # noqa: F401
from .ops import EncodeBuffers, GridSpec, PfnParams, PfnStackParams  # noqa: F401

__version__ = "0.1.0"

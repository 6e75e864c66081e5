"""dvq — B200-native VectorQuantizer + PointNet hot path of D-VQVAE behind the reference's
own module API.  Importing this package loads libdvq_sm100.so; it raises if the library has
not been built (no fallback)."""
from . import _cabi  # noqa: F401  (fails loudly when the CUDA library is missing)
from . import dist  # noqa: F401
from .contact import HandObjectContact, nearest_points  # noqa: F401
from .grasp import GraspGenerator  # noqa: F401
from .host import HostQuantizer  # noqa: F401
from .mano import ManoLayer  # noqa: F401
from .pointnet import PointNetEncoder, STN3d  # noqa: F401
from .quantizer import LazyOneHot, VectorQuantizer  # noqa: F401
from .vqvae import VQVAE  # noqa: F401

__all__ = ["VectorQuantizer", "VQVAE", "PointNetEncoder", "STN3d", "LazyOneHot", "HostQuantizer", "GraspGenerator", "ManoLayer", "HandObjectContact", "nearest_points", "dist"]

"""B200-native point-cloud diffusion sampling hot path (drop-in for the reference's
`PointCloudDiffusion.sample*`, `UNetPointNetLarge.forward`, `metrics.chamfer_distance` and the EMDs of `metrics.py`)."""
from . import _lib
from ._lib import PcdError, build, launch_count
from .diffusion import PointCloudDiffusion
from .latent import (FoldingDecoder, FoldingLayer, LatentDiffusion, PointEncoderEngine, PointNetVAE, SimpleLatentUNetPointNet,
                     SimplePointNetVAE)
from .metrics import (chamfer_distance, chamfer_distance_per_pair, chamfer_matrix, compute_metrics, earth_mover_distance_exact,
                      earth_mover_distance_gpu, emd_matrix, evaluate_sets, set_metrics_from_matrices)
from .networks import PointNetLayer, UNetPointNetLarge
from .voxel import ResidualBlock3D, VAE3DLarge, Vae3dEncoderEngine, Vae3dEngine, voxel_tensor_to_point_clouds
from .parallel import sample_sharded, shard_range
from .synthetic import synthetic_state_dict

__all__ = ["PointCloudDiffusion", "LatentDiffusion", "SimpleLatentUNetPointNet", "SimplePointNetVAE", "PointEncoderEngine", "PointNetVAE", "FoldingDecoder", "FoldingLayer", "UNetPointNetLarge", "PointNetLayer", "chamfer_distance",
           "chamfer_distance_per_pair", "chamfer_matrix", "compute_metrics", "earth_mover_distance_exact", "earth_mover_distance_gpu", "emd_matrix", "evaluate_sets", "set_metrics_from_matrices",
           "VAE3DLarge", "ResidualBlock3D", "Vae3dEngine", "Vae3dEncoderEngine", "voxel_tensor_to_point_clouds",
           "PcdError", "build", "launch_count", "sample_sharded", "shard_range", "synthetic_state_dict"]

"""rpeflow_b200 — the RPEFlow correlation / cost-volume hot path as hand-written sm_100a CUDA kernels.

Public surface (same names as the reference, danqu130/RPEFlow):
  ops         correlation2d, furthest_point_sampling, k_nearest_neighbor      (models/csrc/wrapper.py)
              correlation2d_leaky, warp_correlate                             (RPEFlow_core.py:351,362 fused)
              Correlation2dNCHWFunction — correlation2d's backward on NCHW maps (b200_corr2d_bwd_nchw)
  projection  batch_indexing_channel_{first,last}, grid_sample_wrapper, project_feat_with_nn_corr,
              knn_interpolation, backwarp_3d, backwarp_2d, convex_upsample    (models/utils.py)
              KnnInterpolationFunction, Backwarp2dFunction, ConvexUpsampleFunction, GridSampleFunction,
              BatchIndexingChannelFirstFunction, BatchIndexingChannelLastFunction — their backwards
  pwc3d       Correlation3D, build_pc_pyramid                                 (models/pwc3d_core.py)
              correlation3d, Correlation3DFunction — the same op with a backward (b200_corr3d_bwd)
  pointconv   PointConvDownSampling, PointConvNoSampling                      (models/pointconv.py)
  events      eventsToVoxel, eventsToVoxelInter                               (event_utils.py, dsec.py)
  install     install() — plug all of the above into an unmodified reference checkout
  stack       CostVolumeStack — replays one RPEFlow forward's hot-op census (bench.py's workload)

Importing the package loads rpeflow_b200/libb200flow.so and fails loudly if it is absent: there is no CPU path.
"""
from . import _lib  # noqa: F401  (raises ImportError when the CUDA library is missing)
from .ops import (correlation2d, correlation2d_leaky, warp_correlate, furthest_point_sampling,  # noqa: F401
                  k_nearest_neighbor, squared_distance, CorrelationFunction, Correlation2dNCHWFunction)
from .projection import (batch_indexing_channel_first, batch_indexing_channel_last, grid_sample_wrapper,  # noqa: F401
                         project_feat_with_nn_corr, knn_interpolation, backwarp_3d, backwarp_2d, convex_upsample,
                         KnnInterpolationFunction, Backwarp2dFunction, ConvexUpsampleFunction, GridSampleFunction,
                         BatchIndexingChannelFirstFunction, BatchIndexingChannelLastFunction)
from .pwc3d import (Correlation3D, Correlation3DFunction, build_pc_pyramid, correlation3d,  # noqa: F401
                    correlation3d_forward)
from .pointconv import PointConvDownSampling, PointConvNoSampling, pointconv_forward  # noqa: F401
from .events import eventsToVoxel, eventsToVoxelInter  # noqa: F401

__version__ = "0.1.0"

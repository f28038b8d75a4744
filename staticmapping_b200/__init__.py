"""staticmapping_b200 — B200-native scan matching behind StaticMapping's
registrator::Interface.  The compute lives in libsm_b200.so (hand-written sm_100a CUDA,
C ABI in include/sm_b200.h); this package is the thin host-side mirror used by the tests
and the bench.  There is no CPU fallback."""
from .registrators import (AxisRange, BoundingBoxRemoval, FilterChain, FilterFactory, GroundRemoval, GroundRemoval2, RandomSampler, Range, RangeImage, StatisticRemoval, VoxelGrid,  # noqa: F401
                           AlignBatch, AlignPairs, CalculateNormals, CheckFailure, CreateMatcher, EigenCloud, IcpFast, IcpUsingPointMatcher, InnerCloud,  # noqa: F401
                           Interface, M2dp, MatcherOptions, MrvmSettings, MultiResolutionVoxelMap, matchTwoM2dpDescriptors, MotionCompensation, AverageTransforms, Ndt, NdtWithGicp, Type, VoxelGridFilter, knn1)

__all__ = ["AxisRange", "BoundingBoxRemoval", "FilterChain", "FilterFactory", "GroundRemoval", "GroundRemoval2", "RandomSampler", "Range",
           "RangeImage", "StatisticRemoval", "VoxelGrid", "AlignBatch", "AlignPairs", "CalculateNormals", "CheckFailure", "CreateMatcher", "EigenCloud", "IcpFast", "IcpUsingPointMatcher", "InnerCloud", "Interface", "M2dp", "matchTwoM2dpDescriptors", "Ndt", "NdtWithGicp",
           "MatcherOptions", "MotionCompensation", "MrvmSettings", "MultiResolutionVoxelMap", "AverageTransforms", "Type", "VoxelGridFilter", "knn1"]

"""B200-native A-softmax (SphereFace angular-margin) classification head.

Drop-in for the classifier-FC + softmax-CE slot of medivhna/TF_Face_Toolbox
(nets/sphere.py:84-118, data_parallel.py:203-256): hand-written sm_100a CUDA behind a
C-ABI shared library (include/asoftmax_b200.h), called from Python through ctypes.
"""
from .head import (AdditiveMargin, ASoftmaxHead, ASoftmaxLoss, FocalLoss, FusedOptimizer,  # noqa: F401
                   GraphedASoftmaxStep, LambdaState, asoftmax_head, release_handles)
from .sharded import ShardedASoftmaxHead, shard_bounds  # noqa: F401

__all__ = ["AdditiveMargin", "ASoftmaxHead", "ASoftmaxLoss", "FocalLoss", "FusedOptimizer", "GraphedASoftmaxStep", "LambdaState", "asoftmax_head", "ShardedASoftmaxHead",
           "shard_bounds", "release_handles"]

"""mercer_research_b200 -- B200-native (sm_100a) implementation of rcn's training hot path
(jtstrader/mercer-research): Sobel feature extraction, sigmoid dense layers with quadratic-cost backprop, the
minibatch gradient reduction and the SGD step, behind rcn's own API names.

Compute lives in ``librcn_cuda.so`` (csrc/, C ABI in include/rcn_cuda.h). There is no CPU fallback.
"""
from ._lib import RcnCudaError, load as load_library  # noqa: F401
from .kernel import (Padding, Pooling, SeparableOperator, convolve_2d, convolve_2d_separated, pool_2d, relu,  # noqa: F401
                     sobel_separated)
from .rcn import RCN, RCNLayer  # noqa: F401
from .cnn import SGD, AdamW, Conv, ConvNet, Head, Pool  # noqa: F401

__all__ = ["RCN", "RCNLayer", "ConvNet", "Conv", "Pool", "Head", "SGD", "AdamW", "Padding", "Pooling", "SeparableOperator", "convolve_2d", "convolve_2d_separated",
           "relu", "pool_2d", "sobel_separated", "RcnCudaError", "load_library"]

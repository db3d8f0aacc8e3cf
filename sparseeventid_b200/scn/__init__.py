"""B200-native implementation of the ``sparseconvnet`` module surface (see modules.py)."""
from .config import feature_dtype, get_precision, set_precision
from .core import Metadata, SparseConvNetTensor, prefetch
from .dense_view import SparseDenseTensor
from .functional import prepare_weight_images, release_weight_images
from .modules import (AddTable, AveragePooling, BatchNormalization, BatchNormLeakyReLU, BatchNormReLU, Convolution, Deconvolution,
                      Identity, InputLayer, LeakyReLU, OutputLayer, ReLU, Sequential, Sigmoid, SparseGroupNorm, SparseToDense,
                      SubmanifoldConvolution, Tanh)

__all__ = [
    "AddTable", "AveragePooling", "BatchNormalization", "BatchNormLeakyReLU", "BatchNormReLU", "Convolution", "Deconvolution",
    "Identity", "InputLayer", "LeakyReLU", "OutputLayer", "ReLU", "Sequential", "Sigmoid", "SparseGroupNorm", "SparseToDense",
    "SubmanifoldConvolution", "Tanh", "SparseConvNetTensor", "Metadata", "set_precision", "get_precision",
    "feature_dtype", "SparseDenseTensor", "prefetch", "prepare_weight_images", "release_weight_images",
]

"""B200-native convolutional matching-pursuit engine: drop-in for the MP path of
sbrodeur/hierarchical-sparse-coding (`hsc.modeling`).  CUDA (sm_100a) behind a C ABI
(include/hsc_b200.h); PyTorch only for device memory, streams and torch.distributed."""
from ._native import load_library, HscError, EXPORTED_SYMBOLS   # noqa: F401
from .engine import Engine, EncodeResult, get_engine, engine_dtype   # noqa: F401
from .modeling import (SparseApproximator, ConvolutionalMatchingPursuit, LoCOMP, HierarchicalConvolutionalMatchingPursuit,   # noqa: F401
                       ConvolutionalSparseCoder, HierarchicalConvolutionalSparseCoder, HierarchicalCodes, MultilevelDictionary,
                       ConvolutionalDictionaryLearner, convolve1d, reconstructSignal, normalize)

from .dataset import convertSparseMatricesToEvents, convertEventsToSparseMatrices, encodeResultToEvents   # noqa: F401

__all__ = ['convertSparseMatricesToEvents', 'convertEventsToSparseMatrices', 'Engine', 'EncodeResult', 'get_engine', 'SparseApproximator', 'ConvolutionalMatchingPursuit', 'LoCOMP',
           'HierarchicalConvolutionalMatchingPursuit', 'ConvolutionalSparseCoder', 'HierarchicalConvolutionalSparseCoder',
           'HierarchicalCodes', 'MultilevelDictionary', 'ConvolutionalDictionaryLearner', 'normalize', 'convolve1d', 'reconstructSignal', 'load_library', 'HscError']

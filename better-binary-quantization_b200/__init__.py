"""better-binary-quantization_b200 — B200-native (sm_100a) brute-force quantized search path of
leolee9086/Better-Binary-Quantization, behind the reference's own public API (src/index.ts:20-139).

Only the hot path lives here: csrc/ (CUDA kernels + the C ABI of include/bbq_b200.h), host/ (the
reference-facing operator interface) and bindings/ (the N-API shim + TypeScript glue a Node host uses).
"""
from . import _native
from ._native import build_library
from .host.sharded import ShardedSearcher, broadcast_comm_id, merge_host, shard_bounds
from .host.format import (BbqError, BinarizedByteVectorValues, BinaryQuantizationFormat,
                          GroupBinarizedByteVectorValues, VectorSimilarityFunction)

VERSION = "1.0.0"  # src/index.ts:139

# src/index.ts:47-55
DEFAULT_CONFIG = {"queryBits": 4, "indexBits": 1,
                  "quantizer": {"similarityFunction": VectorSimilarityFunction.COSINE, "lambda": 0.1, "iters": 5}}


def createBinaryQuantizationFormat(config=None, device: int = -1, devices=None) -> BinaryQuantizationFormat:
    """src/index.ts:62-64.  devices: a device group over those GPUs (BinaryQuantizationFormat)."""
    return BinaryQuantizationFormat(config if config is not None else DEFAULT_CONFIG, device=device, devices=devices)


_QUICK_FORMATS = {}


def _quick_format(similarityFunction) -> BinaryQuantizationFormat:
    """The reference builds a fresh format object per quick* call (src/index.ts:76-82,101-107); a format carries no
    state between calls, so one per similarity function is kept: its device context owns the scratch buffers, and
    re-creating those on every call costs more than the 1000-row search the helpers are meant for."""
    fmt = _QUICK_FORMATS.get(similarityFunction)
    if fmt is None:
        fmt = BinaryQuantizationFormat({"quantizer": {"similarityFunction": similarityFunction, "lambda": 0.1, "iters": 5}})
        _QUICK_FORMATS[similarityFunction] = fmt
    return fmt


def quickQuantize(vectors, similarityFunction=VectorSimilarityFunction.COSINE):
    """src/index.ts:72-85"""
    return _quick_format(similarityFunction).quantizeVectors(vectors)


def quickSearch(queryVector, targetVectors, k, similarityFunction=VectorSimilarityFunction.COSINE):
    """src/index.ts:95-111 — like the reference, re-quantises the corpus on every call."""
    fmt = _quick_format(similarityFunction)
    qv = fmt.quantizeVectors(targetVectors)["quantizedVectors"]
    return fmt.searchNearestNeighbors(queryVector, qv, k)


def getOversampledTopKWithSort(query, quantizedVectors, vectors, k, oversampleFactor, format):
    """src/topKSelector.ts:90-114 (same argument order).  `vectors` (the original rows) are attached to the device
    index on first use.  -> [{index, quantizedScore, trueScore}] by trueScore descending."""
    if not getattr(quantizedVectors, "_rows_attached", False):
        format.attachOriginalVectors(quantizedVectors, vectors)
        quantizedVectors._rows_attached = True
    import numpy as _np
    i, qs, ts = format.searchOversampledBatch(_np.asarray(query, _np.float32)[None, :], quantizedVectors, k,
                                              oversampleFactor)
    return [{"index": int(a), "quantizedScore": float(b), "trueScore": float(c)} for a, b, c in zip(i[0], qs[0], ts[0])]


getOversampledTopKWithHeap = getOversampledTopKWithSort  # :29-78 — same set unless true scores tie at the k-th place


__all__ = ["BinaryQuantizationFormat", "BinarizedByteVectorValues", "GroupBinarizedByteVectorValues", "VectorSimilarityFunction", "BbqError",
           "createBinaryQuantizationFormat", "quickQuantize", "quickSearch", "DEFAULT_CONFIG", "VERSION",
           "build_library", "ShardedSearcher", "shard_bounds", "merge_host", "broadcast_comm_id", "getOversampledTopKWithSort",
           "getOversampledTopKWithHeap"]

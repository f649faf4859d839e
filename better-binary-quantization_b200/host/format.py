"""Host-side mirror of the reference's operator interface for the search path (Python stand-in for the
TypeScript layer, which cannot run here: no Node in the image — see INTEGRATION.md for the real TS/N-API
binding).  Same names, argument meaning and error behaviour as the reference:

  BinaryQuantizationFormat            src/binaryQuantizationFormat.ts:132-412
    .quantizeVectors(vectors)         :165-263  -> {quantizedVectors, queryQuantizer}
    .quantizeQueryVector(q, centroid) :271-299
    .searchNearestNeighbors(q, t, k)  :308-412  -> [{index, score}] descending
  BinarizedByteVectorValues           src/types.ts:32-49 (an opaque device handle here)
  VectorSimilarityFunction            src/types.ts:9-13

Everything numeric happens in libbbq_b200.so on the GPU; this file only marshals and maps errors.
"""
from __future__ import annotations

import ctypes as C
import math
import os
from typing import List, Optional, Sequence

import numpy as np

from .. import _native

QUERY_BITS = 4   # src/constants.ts:9
INDEX_BITS = 1   # src/constants.ts:14


class VectorSimilarityFunction:
    EUCLIDEAN = "EUCLIDEAN"
    COSINE = "COSINE"
    MAXIMUM_INNER_PRODUCT = "MAXIMUM_INNER_PRODUCT"


_SIM_CODE = {"EUCLIDEAN": 0, "COSINE": 1, "MAXIMUM_INNER_PRODUCT": 2}

# status -> the reference's message (file:line in include/bbq_b200.h)
def _message(status: int, vec: int, pos: int, what: str) -> str:
    return {
        1: "queryBits必须在1-8之间",
        2: "indexBits必须在1-8之间",
        3: "向量集合不能为空",
        7: "k值不能为负数",
    }.get(status) or {
        ("build", 5): f"向量 {vec} 位置 {pos} 包含NaN值",
        ("build", 6): f"向量 {vec} 位置 {pos} 包含Infinity值",
        ("search", 5): f"向量位置 {pos} 包含NaN值",
        ("search", 6): f"向量位置 {pos} 包含Infinity值",
        ("search", 4): "查询向量维度与目标向量维度不匹配",
    }.get((what, status)) or _native.load().bbq_last_error().decode()


class BbqError(Exception):
    """`throw new Error(msg)` of the reference; .status is the C-ABI status code."""

    def __init__(self, status: int, message: str):
        super().__init__(message)
        self.status = status


def _check(status: int, what: str = ""):
    if status != 0:
        v, p = C.c_int64(-1), C.c_int64(-1)
        _native.load().bbq_last_error_pos(C.byref(v), C.byref(p))
        raise BbqError(status, _message(status, v.value, p.value, what))


def _as_matrix(vectors) -> np.ndarray:
    """Float32Array[] -> contiguous [n, dim] f32; ragged input raises the reference's message (:190-192)."""
    if isinstance(vectors, np.ndarray) and vectors.ndim == 2:
        return np.ascontiguousarray(vectors, dtype=np.float32)
    rows = [np.asarray(v, dtype=np.float32).ravel() for v in vectors]
    if not rows:
        return np.empty((0, 0), np.float32)
    d = rows[0].size
    for i, r in enumerate(rows[1:], 1):
        if r.size != d:
            raise BbqError(4, f"向量 {i} 维度 {r.size} 与第一个向量维度 {d} 不匹配")
    return np.ascontiguousarray(np.stack(rows), dtype=np.float32)


class _VectorValues:
    """The read-only members of src/types.ts:32-49 over a device index, whatever its handle type.
    size()/dimension()/getCentroid() answer from cached host metadata; vectorValue()/getCorrectiveTerms() do a lazy
    device->host copy (cold path, SURVEY §8b) through _export_rows, which each handle type provides."""

    def _read_meta(self, size, dim, centroid):
        self._n = int(size(self._h))
        self._dim = int(dim(self._h))
        c = np.empty(self._dim, np.float32)
        cdp = C.c_double()
        _check(centroid(self._h, c.ctypes.data, C.byref(cdp)))
        self._centroid, self._cdp = c, cdp.value

    def dimension(self) -> int:
        return self._dim

    def size(self) -> int:
        return self._n

    def getCentroid(self) -> np.ndarray:
        return self._centroid

    def getCentroidDP(self, queryVector=None) -> float:
        if queryVector is not None:  # src/binaryQuantizationFormat.ts:113-117 (not used by search)
            q = np.asarray(queryVector, np.float32).astype(np.float64)
            s = 0.0
            for a, b in zip(q, self._centroid.astype(np.float64)):
                s += a * b
            return s
        return self._cdp

    def _export(self, ord_: int, count: int = 1):
        if ord_ < 0 or ord_ + count > self._n:
            raise BbqError(10, f"向量索引 {ord_} 不存在")
        # indexBits == 1: packed MSB-first rows of ceil(dim/8) bytes; otherwise dim unpacked codes per row, as
        # BinarizedByteVectorValuesImpl holds them (src/binaryQuantizationFormat.ts:221-249)
        p = (self._dim + 7) // 8 if self._fmt.config["indexBits"] == 1 else self._dim
        packed = np.empty((count, p), np.uint8)
        corr = np.empty((count, 4), np.float64)
        self._export_rows(ord_, count, packed.ctypes.data, corr.ctypes.data)
        return packed, corr

    def vectorValue(self, ord_: int) -> np.ndarray:
        return self._export(ord_)[0][0]

    def getUnpackedVector(self, ord_: int) -> np.ndarray:
        if ord_ < 0 or ord_ >= self._n:
            raise BbqError(10, f"未打包向量索引 {ord_} 不存在")
        v = self.vectorValue(ord_)
        return np.unpackbits(v)[: self._dim] if self._fmt.config["indexBits"] == 1 else v

    def getCorrectiveTerms(self, ord_: int) -> dict:
        c = self._export(ord_)[1][0]
        return {"lowerInterval": c[0], "upperInterval": c[1], "additionalCorrection": c[2],
                "quantizedComponentSum": c[3]}

    def exportAll(self):
        """(packed u8[n, ceil(dim/8)], corr f64[n,4]) — test/diagnostic convenience."""
        return self._export(0, self._n)


class BinarizedByteVectorValues(_VectorValues):
    """Device-resident index shard on one GPU (a bbq_index)."""

    def __init__(self, fmt: "BinaryQuantizationFormat", handle):
        self._fmt = fmt
        self._h = handle
        L = _native.load()
        self._read_meta(L.bbq_index_size, L.bbq_index_dim, L.bbq_index_centroid)

    def __del__(self):
        try:
            if self._h is not None:
                _native.load().bbq_index_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def _export_rows(self, first, count, packed, corr):
        _check(_native.load().bbq_index_export(self._h, first, count, packed, corr))


class GroupBinarizedByteVectorValues(_VectorValues):
    """An index of a device group: one row shard per GPU of the group (a bbq_group_index), the same read-only members
    as BinarizedByteVectorValues.  vectorValue()/getCorrectiveTerms() read from the shard that holds the row.  It is
    not a BinarizedByteVectorValues: its handle never reaches a bbq_index_* entry (_index refuses it)."""

    def __init__(self, fmt: "BinaryQuantizationFormat", handle):
        self._fmt = fmt
        self._h = handle
        L = _native.load()
        self._read_meta(L.bbq_group_index_size, L.bbq_group_index_dim, L.bbq_group_index_centroid)

    def __del__(self):
        try:
            if self._h is not None:
                _native.load().bbq_group_index_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def _export_rows(self, first, count, packed, corr):
        _check(_native.load().bbq_group_index_export(self._h, first, count, packed, corr))


def _index(targetVectors):
    """The bbq_index* of a one-GPU index, for the entries that take one.  A device group's index is another type in C
    (bbq_group_index*): it is refused here, never handed over."""
    if isinstance(targetVectors, GroupBinarizedByteVectorValues):
        raise BbqError(10, "this member takes an index on one GPU; a device group's index is served by quantizeVectors, "
                           "searchNearestNeighbors, searchBatch, attachOriginalVectors, searchOversampledBatch, saveIndex "
                           "and its own members")
    return targetVectors._h


class BinaryQuantizationFormat:
    def __init__(self, config: dict, device: int = -1, devices: Optional[Sequence[int]] = None):
        """devices: the GPUs of a device group (bbq_group_create): one process drives all of them, every index is split
        into one row shard per GPU, and builds, searches, re-ranks and images run on all of them at once.
        quantizeQueryVector and computeQuantizationAccuracy run on the group's first GPU."""
        q = config.get("quantizer") or {}
        self.config = {"queryBits": QUERY_BITS, "indexBits": INDEX_BITS, **config}
        cfg = _native.BbqConfig()
        cfg.query_bits = int(self.config["queryBits"]) if 0 <= self.config["queryBits"] < 2**31 else 0
        cfg.index_bits = int(self.config["indexBits"]) if 0 <= self.config["indexBits"] < 2**31 else 0
        # src/optimizedScalarQuantizer.ts:48-50 defaults
        self._sim = q.get("similarityFunction", VectorSimilarityFunction.EUCLIDEAN)
        cfg.similarity = _SIM_CODE[self._sim]
        cfg.lambda_ = float(q.get("lambda", 0.1))
        cfg.iters = int(q.get("iters", 5))
        cfg.device = device
        self._ctx = C.c_void_p()
        self._group = None
        L = _native.load()
        if devices is None:
            _check(L.bbq_create(C.byref(cfg), C.byref(self._ctx)))
            return
        devs = (C.c_int32 * max(len(devices), 1))(*[int(d) for d in devices])
        group = C.c_void_p()
        _check(L.bbq_group_create(C.byref(cfg), devs, len(devices), C.byref(group)))
        self._group = group
        self._in_group = True
        self._ctx = C.c_void_p(L.bbq_group_context(group, 0))   # owned by the group

    def __del__(self):
        try:
            if getattr(self, "_group", None):
                _native.load().bbq_group_destroy(self._group)
                self._group = None
            elif getattr(self, "_ctx", None) and not getattr(self, "_in_group", False):
                _native.load().bbq_destroy(self._ctx)
            self._ctx = None
        except Exception:
            pass

    def devices(self) -> List[int]:
        """The GPUs of this format's device group ([] without one)."""
        if not self._group:
            return []
        L = _native.load()
        n = C.c_uint32(0)
        _check(L.bbq_group_info(self._group, C.byref(n), None))
        out = (C.c_int32 * n.value)()
        _check(L.bbq_group_info(self._group, C.byref(n), out))
        return list(out)

    def groupContext(self, rank: int) -> int:
        """The context of rank `rank` of the device group (bbq_group_context), for statistics."""
        return _native.load().bbq_group_context(self._group, rank)

    def _not_sharded(self, sharded: bool):
        if sharded and self._group:
            raise BbqError(10, "a device-group format is already sharded over its GPUs: sharded=True does not apply")

    def _one_gpu(self, member: str):
        """Device-pointer, streaming, shard-bootstrap and debug members exist for one GPU only: on a device-group format
        they would act on its first GPU's context alone, so they are refused."""
        if self._group:
            raise BbqError(10, f"{member} is not available on a device-group format")

    def getConfig(self) -> dict:
        return dict(self.config)

    # -- index build ----------------------------------------------------------------------------------
    def quantizeVectors(self, vectors, centroid: Optional[np.ndarray] = None, sharded: bool = False) -> dict:
        """sharded=True: this rank's rows of a corpus split over the communicator in rank order (bbq_index_build_sharded,
        collective); the rank may hold no rows.  Without a centroid every rank gets the reference-order centroid of the
        whole corpus, and its shard (base set) equals its rows of the whole-corpus build."""
        self._not_sharded(sharded)
        if not sharded and (vectors is None or len(vectors) == 0):
            raise BbqError(3, "向量集合不能为空")
        m = _as_matrix(vectors if vectors is not None else [])
        h = C.c_void_p()
        cen = np.ascontiguousarray(centroid, np.float32) if centroid is not None else None
        L = _native.load()
        if self._group:
            _check(L.bbq_group_index_build(self._group, m.ctypes.data, m.shape[0], m.shape[1],
                                           cen.ctypes.data if cen is not None else None, C.byref(h)), "build")
            return {"quantizedVectors": GroupBinarizedByteVectorValues(self, h), "queryQuantizer": self}
        if sharded:
            dim = m.shape[1] if m.shape[0] else (cen.size if cen is not None else 0)
            _check(L.bbq_index_build_sharded(self._ctx, m.ctypes.data, m.shape[0], dim,
                                             cen.ctypes.data if cen is not None else None, C.byref(h)), "build")
        else:
            _check(L.bbq_index_build(self._ctx, m.ctypes.data, m.shape[0], m.shape[1],
                                     cen.ctypes.data if cen is not None else None, C.byref(h)), "build")
        # (the reference hands out its OptimizedScalarQuantizer helper as queryQuantizer, :261, and so does the TypeScript
        # drop-in; this Python stand-in has no such host-side object: the format itself quantises queries)
        return {"quantizedVectors": BinarizedByteVectorValues(self, h), "queryQuantizer": self}

    def quantizeVectorsDevice(self, d_rows_ptr: int, n: int, dim: int, centroid: Optional[np.ndarray] = None,
                              sharded: bool = False):
        """Rows already in device memory (e.g. a torch tensor's data_ptr()).  sharded=True: as quantizeVectors
        (bbq_index_build_sharded_device, collective)."""
        self._one_gpu("quantizeVectorsDevice")
        self._not_sharded(sharded)
        h = C.c_void_p()
        cen = np.ascontiguousarray(centroid, np.float32) if centroid is not None else None
        L = _native.load()
        fn = L.bbq_index_build_sharded_device if sharded else L.bbq_index_build_device
        _check(fn(self._ctx, d_rows_ptr or None, n, dim, cen.ctypes.data if cen is not None else None, C.byref(h)),
               "build")
        return {"quantizedVectors": BinarizedByteVectorValues(self, h), "queryQuantizer": self}

    def accumulateCentroid(self, running: np.ndarray, rowsBefore: int, rows=None, d_rows_ptr: int = 0, n: int = 0):
        """The reference centroid's running sum (f32[dim], updated in place and returned) continued over the rows that
        follow the corpus's first rowsBefore rows: host `rows`, or n device rows at d_rows_ptr
        (bbq_centroid_accumulate / _device).  rowsBefore == 0 starts the corpus."""
        self._one_gpu("accumulateCentroid")
        if running.dtype != np.float32 or not running.flags.c_contiguous:
            raise BbqError(10, "running must be a contiguous float32 array")
        L = _native.load()
        if rows is not None:
            m = _as_matrix(rows)
            if m.shape[0] and m.shape[1] != running.size:
                raise BbqError(4, "向量维度不匹配")
            _check(L.bbq_centroid_accumulate(self._ctx, m.ctypes.data, m.shape[0], running.size, rowsBefore,
                                             running.ctypes.data), "build")
        else:
            _check(L.bbq_centroid_accumulate_device(self._ctx, d_rows_ptr or None, n, running.size, rowsBefore,
                                                    running.ctypes.data), "build")
        return running

    @staticmethod
    def finishCentroid(running, nTotal: int) -> np.ndarray:
        """f32(running / N) in f64 (bbq_centroid_finish): the centroid bbq_index_build computes for N rows."""
        r = np.ascontiguousarray(running, np.float32)
        out = np.empty(r.size, np.float32)
        _check(_native.load().bbq_centroid_finish(r.ctypes.data, r.size, nTotal, out.ctypes.data), "build")
        return out

    def reserveIndex(self, capacity: int, dim: int, centroid) -> BinarizedByteVectorValues:
        """Streaming build (bbq_index_reserve): explicit centroid, rows appended chunk by chunk."""
        self._one_gpu("reserveIndex")
        cen = np.ascontiguousarray(centroid, np.float32)
        h = C.c_void_p()
        _check(_native.load().bbq_index_reserve(self._ctx, capacity, dim, cen.ctypes.data, C.byref(h)), "build")
        return BinarizedByteVectorValues(self, h)

    def appendRows(self, targetVectors: BinarizedByteVectorValues, rows=None, d_rows_ptr: int = 0, n: int = 0):
        self._one_gpu("appendRows")
        L = _native.load()
        if rows is not None:
            m = _as_matrix(rows)
            _check(L.bbq_index_append(_index(targetVectors), m.ctypes.data, m.shape[0]), "build")
        else:
            _check(L.bbq_index_append_device(_index(targetVectors), d_rows_ptr, n), "build")
        targetVectors._n = int(L.bbq_index_size(_index(targetVectors)))

    def adoptQuantized(self, packed, corr4, centroid) -> BinarizedByteVectorValues:
        """Index quantised elsewhere (e.g. by the reference): bbq_index_from_quantized."""
        packed = np.ascontiguousarray(packed, np.uint8)
        corr4 = np.ascontiguousarray(corr4, np.float64)
        centroid = np.ascontiguousarray(centroid, np.float32)
        h = C.c_void_p()
        if self._group:
            _check(_native.load().bbq_group_index_from_quantized(self._group, packed.ctypes.data, corr4.ctypes.data,
                                                                 centroid.ctypes.data, packed.shape[0], centroid.size,
                                                                 C.byref(h)), "build")
            return GroupBinarizedByteVectorValues(self, h)
        _check(_native.load().bbq_index_from_quantized(self._ctx, packed.ctypes.data, corr4.ctypes.data,
                                                       centroid.ctypes.data, packed.shape[0], centroid.size,
                                                       C.byref(h)), "build")
        return BinarizedByteVectorValues(self, h)

    # -- index image on disk (serializeVectorData / deserializeVectorData, :483-560) ----------------------
    @staticmethod
    def _image_paths(prefix: str):
        # FILE_EXTENSIONS, src/constants.ts:52-57
        return (os.fsencode(prefix + ".veb"), os.fsencode(prefix + ".vemb"))

    def saveIndex(self, targetVectors: BinarizedByteVectorValues, prefix: str, sharded: bool = False) -> None:
        """Writes <prefix>.veb (vector data) and <prefix>.vemb (metadata + centroid): bbq_index_save.  sharded=True: one
        image of all row shards of the communicator, each rank writing its own rows (bbq_index_save_sharded,
        collective); the files equal those of one index holding the whole corpus."""
        self._not_sharded(sharded)
        veb, vemb = self._image_paths(prefix)
        L = _native.load()
        if isinstance(targetVectors, GroupBinarizedByteVectorValues):
            fn = L.bbq_group_index_save
        else:
            fn = L.bbq_index_save_sharded if sharded else L.bbq_index_save
        _check(fn(targetVectors._h, veb, vemb), "build")

    def loadIndex(self, prefix: str, sharded: bool = False) -> BinarizedByteVectorValues:
        """Reads an image written by saveIndex straight into device memory: bbq_index_load.  sharded=True: this rank's
        row range of the image (shard_bounds), with its base set (bbq_index_load_sharded, collective)."""
        self._not_sharded(sharded)
        veb, vemb = self._image_paths(prefix)
        h = C.c_void_p()
        L = _native.load()
        if self._group:
            _check(L.bbq_group_index_load(self._group, veb, vemb, C.byref(h)), "build")
            return GroupBinarizedByteVectorValues(self, h)
        fn = L.bbq_index_load_sharded if sharded else L.bbq_index_load
        _check(fn(self._ctx, veb, vemb, C.byref(h)), "build")
        return BinarizedByteVectorValues(self, h)

    def loadIndexRows(self, prefix: str, first: int, count: int):
        """Rows [first, first + count) of an image as an index whose base is `first` (bbq_index_load_rows, not
        collective) -> (index, the five partial section checksums of the rows loaded)."""
        self._one_gpu("loadIndexRows")
        veb, vemb = self._image_paths(prefix)
        h = C.c_void_p()
        part = (C.c_uint64 * 5)()
        _check(_native.load().bbq_index_load_rows(self._ctx, veb, vemb, first, count, C.byref(h), part), "build")
        return BinarizedByteVectorValues(self, h), [int(x) for x in part]

    def writeIndexRows(self, shard: BinarizedByteVectorValues, prefix: str, totalRows: int):
        """This shard's rows at rows [base, base + size) of an image of totalRows rows (bbq_index_write_rows)
        -> the five partial section checksums of the rows written."""
        self._one_gpu("writeIndexRows")
        veb, _ = self._image_paths(prefix)
        part = (C.c_uint64 * 5)()
        _check(_native.load().bbq_index_write_rows(_index(shard), veb, totalRows, part), "build")
        return [int(x) for x in part]

    def writeIndexMeta(self, shard: BinarizedByteVectorValues, prefix: str, totalRows: int, checksums) -> None:
        """<prefix>.vemb for an image of totalRows rows whose sections have the given checksums (the sums mod 2^64 of
        every shard's partials) and this shard's centroid (bbq_index_write_meta)."""
        self._one_gpu("writeIndexMeta")
        _, vemb = self._image_paths(prefix)
        sums = (C.c_uint64 * 5)(*[int(x) & 0xFFFFFFFFFFFFFFFF for x in checksums])
        _check(_native.load().bbq_index_write_meta(_index(shard), vemb, totalRows, sums), "build")

    def setBase(self, targetVectors: BinarizedByteVectorValues, base: int) -> None:
        """Global row id of this shard's row 0 (bbq_index_set_base)."""
        self._one_gpu("setBase")
        _check(_native.load().bbq_index_set_base(_index(targetVectors), base))

    # -- query side -------------------------------------------------------------------------------------
    def quantizeQueryVector(self, queryVector, centroid) -> dict:
        """src/binaryQuantizationFormat.ts:271-299.  With a centroid ARRAY (the reference signature) this is the class
        member as written: a COSINE query is normalised once, then scalarQuantize(queryBits) (bbq_quantize_query).
        With a device index handle instead of the centroid it is the query quantisation of the SEARCH path
        (searchNearestNeighbors normalises at :337 and again at :279 — twice), the parity tap the tests compare."""
        q = np.ascontiguousarray(queryVector, np.float32)
        codes = np.empty(q.size, np.uint8)
        corr = np.empty(4, np.float64)
        if isinstance(centroid, (BinarizedByteVectorValues, GroupBinarizedByteVectorValues)):
            _check(_native.load().bbq_debug_quantize_query(_index(centroid), q.ctypes.data, codes.ctypes.data,
                                                           corr.ctypes.data), "search")
        else:
            cen = np.ascontiguousarray(centroid, np.float32)
            if cen.size != q.size:
                raise BbqError(4, "查询向量维度与目标向量维度不匹配")
            _check(_native.load().bbq_quantize_query(self._ctx, q.ctypes.data, cen.ctypes.data, q.size,
                                                     codes.ctypes.data, corr.ctypes.data), "search")
        return {"quantizedQuery": codes,
                "queryCorrections": {"lowerInterval": corr[0], "upperInterval": corr[1],
                                     "additionalCorrection": corr[2], "quantizedComponentSum": corr[3]}}

    def computeQuantizationAccuracy(self, originalVectors, queryVectors, targetOrd: int = 0) -> dict:
        """src/binaryQuantizationFormat.ts:420-475 + src/binaryQuantizedScorer.ts:524-617 on the device
        (bbq_quantization_accuracy): every query scored against row `targetOrd` (the reference: 0) through the
        single-vector quantised scorer and exactly; -> {meanError, maxError, minError, stdError, correlation}."""
        if originalVectors is None or len(originalVectors) == 0:
            raise BbqError(3, "原始向量集合不能为空")
        if queryVectors is None or len(queryVectors) == 0:
            raise BbqError(3, "查询向量集合不能为空")
        if len(originalVectors) != len(queryVectors):
            raise BbqError(10, "原始向量集合和查询向量集合长度不匹配")
        if self.config["queryBits"] not in (1, 4):   # computeQuantizedScore, src/binaryQuantizedScorer.ts:96
            raise BbqError(9, f"不支持的查询位数: {self.config['queryBits']}，只支持1位和4位")
        m, q = _as_matrix(originalVectors), _as_matrix(queryVectors)
        if q.shape[1] != m.shape[1]:
            raise BbqError(4, "向量维度不匹配")
        out = np.empty(5, np.float64)
        _check(_native.load().bbq_quantization_accuracy(self._ctx, m.ctypes.data, q.ctypes.data, m.shape[0], m.shape[1],
                                                        targetOrd, out.ctypes.data), "build")
        return dict(zip(("meanError", "maxError", "minError", "stdError", "correlation"), out.tolist()))

    def serializeVectorData(self, vectors) -> dict:
        """src/binaryQuantizationFormat.ts:483-525: quantise (on the device) and return the reference's
        {vectorData: [VectorDataFormat], metadata: MetadataFormat} objects (src/types.ts:78-113).  binaryValues is
        the packed MSB-first row (the reference re-packs an already packed row here, which yields ceil(P/8) bytes of
        no use: the working form is kept).  For indexes that should reach a disk use saveIndex."""
        qv = self.quantizeVectors(vectors)["quantizedVectors"]
        packed, corr = qv.exportAll()
        cen = qv.getCentroid()
        data = [{"binaryValues": packed[i], "lowerInterval": corr[i, 0], "upperInterval": corr[i, 1],
                 "additionalCorrection": corr[i, 2], "quantizedComponentSum": corr[i, 3]} for i in range(qv.size())]
        meta = {"fieldNumber": 0, "vectorEncodingOrdinal": 0, "vectorSimilarityOrdinal": 0, "dimensions": int(cen.size),
                "vectorDataOffset": 0, "vectorDataLength": 0, "vectorCount": qv.size(), "centroid": cen,
                "centroidSquareMagnitude": qv.getCentroidDP()}
        return {"vectorData": data, "metadata": meta}

    def deserializeVectorData(self, vectorData, metadata) -> BinarizedByteVectorValues:
        """src/binaryQuantizationFormat.ts:533-560: back to a (device-resident) BinarizedByteVectorValues."""
        packed = np.stack([np.asarray(d["binaryValues"], np.uint8) for d in vectorData])
        corr = np.array([[d["lowerInterval"], d["upperInterval"], d["additionalCorrection"],
                          d["quantizedComponentSum"]] for d in vectorData], np.float64)
        return self.adoptQuantized(packed, corr, metadata["centroid"])

    # -- search -----------------------------------------------------------------------------------------
    def searchNearestNeighbors(self, queryVector, targetVectors: BinarizedByteVectorValues, k: int) -> List[dict]:
        if queryVector is None:
            raise BbqError(8, "查询向量不能为空")
        if targetVectors is None:
            raise BbqError(8, "目标向量集合不能为空")
        if k < 0:
            raise BbqError(7, "k值不能为负数")
        k = int(math.ceil(k))      # a fractional k: the reference's heap loop (`size() < k2`) ends up with ceil(k) results
        q = np.ascontiguousarray(queryVector, np.float32).ravel()
        if q.size != targetVectors.dimension():
            raise BbqError(4, "查询向量维度与目标向量维度不匹配")
        idx, sc = self.searchBatch(q[None, :], targetVectors, k)
        return [{"index": int(i), "score": float(s)} for i, s in zip(idx[0], sc[0])]

    def searchBatch(self, queries, targetVectors: BinarizedByteVectorValues, k: int, sharded: bool = False):
        """Additive batched entry (SURVEY §8b): row i == searchNearestNeighbors(queries[i]).
        -> (idx i32[nq, min(k,n)], score f32[nq, min(k,n)]).  sharded=True: over all row shards of the communicator
        (bbq_search_sharded, collective; n = the rows of all shards), the same lists on every rank."""
        if k < 0:
            raise BbqError(7, "k值不能为负数")
        qs = np.ascontiguousarray(queries, np.float32)
        if qs.ndim != 2 or qs.shape[1] != targetVectors.dimension():
            raise BbqError(4, "查询向量维度与目标向量维度不匹配")
        nq = qs.shape[0]
        kk = min(k, targetVectors.size())
        idx = np.empty((nq, max(k, 1)), np.int32)
        sc = np.empty((nq, max(k, 1)), np.float32)
        cnt = C.c_uint32(0)
        L = _native.load()
        self._not_sharded(sharded)
        if isinstance(targetVectors, GroupBinarizedByteVectorValues):
            fn = L.bbq_group_search
        else:
            fn = L.bbq_search_sharded if sharded else L.bbq_search
        _check(fn(targetVectors._h, qs.ctypes.data, nq, k, idx.ctypes.data, sc.ctypes.data, C.byref(cnt)), "search")
        assert sharded or cnt.value == (kk if nq else 0) or k == 0
        return idx[:, :cnt.value].copy(), sc[:, :cnt.value].copy()

    # -- oversampled search + exact re-rank (src/topKSelector.ts) -------------------------------------------
    def attachOriginalVectors(self, targetVectors: BinarizedByteVectorValues, vectors):
        """Keeps the original f32 rows on the device next to the index (needed by the exact re-rank)."""
        m = _as_matrix(vectors)
        if m.shape[0] != targetVectors.size() or m.shape[1] != targetVectors.dimension():
            raise BbqError(4, "向量维度不匹配")
        L = _native.load()
        fn = L.bbq_group_index_attach_rows if isinstance(targetVectors, GroupBinarizedByteVectorValues) else L.bbq_index_attach_rows
        _check(fn(targetVectors._h, m.ctypes.data), "build")

    def attachOriginalVectorsDevice(self, targetVectors: BinarizedByteVectorValues, d_rows_ptr: int):
        """Same, rows already in device memory ([size, dimension] f32, e.g. a torch tensor's data_ptr())."""
        self._one_gpu("attachOriginalVectorsDevice")
        _check(_native.load().bbq_index_attach_rows_device(_index(targetVectors), d_rows_ptr), "build")

    def searchOversampledBatch(self, queries, targetVectors: BinarizedByteVectorValues, k: int, oversampleFactor: int,
                               sharded: bool = False):
        """-> (idx i32[nq, kk], quantizedScore f32[nq, kk], trueScore f64[nq, kk]).  sharded=True: over all row shards
        of the communicator (bbq_search_rerank_sharded, collective), the same lists on every rank."""
        qs = np.ascontiguousarray(queries, np.float32)
        if qs.ndim != 2 or qs.shape[1] != targetVectors.dimension():
            raise BbqError(4, "查询向量维度与目标向量维度不匹配")
        nq = qs.shape[0]
        idx = np.empty((nq, max(k, 1)), np.int32)
        qsc = np.empty((nq, max(k, 1)), np.float32)
        tsc = np.empty((nq, max(k, 1)), np.float64)
        cnt = C.c_uint32(0)
        L = _native.load()
        self._not_sharded(sharded)
        if isinstance(targetVectors, GroupBinarizedByteVectorValues):
            fn = L.bbq_group_search_rerank
        else:
            fn = L.bbq_search_rerank_sharded if sharded else L.bbq_search_rerank
        _check(fn(targetVectors._h, qs.ctypes.data, nq, k, oversampleFactor, idx.ctypes.data, qsc.ctypes.data,
                  tsc.ctypes.data, C.byref(cnt)), "search")
        n = cnt.value
        return idx[:, :n].copy(), qsc[:, :n].copy(), tsc[:, :n].copy()

    def rerankOwnedDevice(self, targetVectors: BinarizedByteVectorValues, d_queries_ptr: int, nq: int,
                          d_cand_idx_ptr: int, m: int, d_true_bits_ptr: int, stream: int = 0):
        """bbq_rerank_owned_device: [nq][m] u64 = this shard's exact-score bits for the candidates it holds, else 0."""
        self._one_gpu("rerankOwnedDevice")
        _check(_native.load().bbq_rerank_owned_device(_index(targetVectors), d_queries_ptr, nq, d_cand_idx_ptr, m,
                                                      d_true_bits_ptr, stream or None), "search")

    # -- parity taps (tests) ------------------------------------------------------------------------------
    def debugQcDist(self, queryVector, targetVectors: BinarizedByteVectorValues) -> np.ndarray:
        self._one_gpu("debugQcDist")
        q = np.ascontiguousarray(queryVector, np.float32)
        out = np.empty(targetVectors.size(), np.int32)
        _check(_native.load().bbq_debug_qcdist(_index(targetVectors), q.ctypes.data, out.ctypes.data), "search")
        return out

    def debugQcDistBatch(self, queries, targetVectors: BinarizedByteVectorValues) -> np.ndarray:
        """The integer dots of the TENSOR-CORE scan (tcgen05 accumulators) for a query batch: int32 [nq, n]."""
        self._one_gpu("debugQcDistBatch")
        qs = np.ascontiguousarray(queries, np.float32)
        out = np.empty((qs.shape[0], targetVectors.size()), np.int32)
        _check(_native.load().bbq_debug_qcdist_batch(_index(targetVectors), qs.ctypes.data, qs.shape[0], out.ctypes.data),
               "search")
        return out

    def debugScores(self, queryVector, targetVectors: BinarizedByteVectorValues) -> np.ndarray:
        self._one_gpu("debugScores")
        q = np.ascontiguousarray(queryVector, np.float32)
        out = np.empty(targetVectors.size(), np.float32)
        _check(_native.load().bbq_debug_scores(_index(targetVectors), q.ctypes.data, out.ctypes.data), "search")
        return out

    def stats(self) -> dict:
        s = _native.BbqStats()
        _check(_native.load().bbq_get_stats(self._ctx, C.byref(s)))
        return {"kernel_launches": s.kernel_launches, "last_candidates": s.last_candidates,
                "last_path": s.last_path, "last_overflow": s.last_overflow, "last_engine": s.last_engine,
                "scan_launches": s.scan_launches,
                "scan_ms": s.scan_ms, "quantize_ms": s.quantize_ms, "select_ms": s.select_ms, "sample_ms": s.sample_ms,
                "mma_n_tile": s.mma_n_tile, "mma_passes": s.mma_passes, "mma_layout": s.mma_layout, "graph_replays": s.graph_replays}

    def setProfiling(self, enabled: bool):
        _check(_native.load().bbq_set_profiling(self._ctx, 1 if enabled else 0))

    def resetProfiling(self):
        _check(_native.load().bbq_reset_profiling(self._ctx))

    # -- device-resident entry points (plumbing for sharded search: torch tensors' data_ptr()) ------------
    def searchDevice(self, d_queries_ptr: int, nq: int, targetVectors: BinarizedByteVectorValues, k: int,
                     d_out_idx_ptr: int, d_out_score_ptr: int, stream: int = 0):
        self._one_gpu("searchDevice")
        _check(_native.load().bbq_search_device(_index(targetVectors), d_queries_ptr, nq, k, d_out_idx_ptr,
                                                d_out_score_ptr, stream or None), "search")

    # -- sharded search: the exchange lives in the library (bbq_comm_*, one NCCL all-gather of 64-bit keys) -----
    @staticmethod
    def commUniqueId() -> bytes:
        buf = (C.c_uint8 * 128)()
        _check(_native.load().bbq_comm_unique_id(buf))
        return bytes(buf)

    def commInit(self, comm_id: bytes, rank: int, world: int):
        self._one_gpu("commInit")
        buf = (C.c_uint8 * 128).from_buffer_copy(comm_id)
        _check(_native.load().bbq_comm_init(self._ctx, buf, rank, world))

    def commDestroy(self):
        self._one_gpu("commDestroy")
        _check(_native.load().bbq_comm_destroy(self._ctx))

    def commInfo(self) -> dict:
        r, w, v = C.c_int(), C.c_int(), C.c_int()
        _check(_native.load().bbq_comm_info(self._ctx, C.byref(r), C.byref(w), C.byref(v)))
        return {"rank": r.value, "world": w.value, "nccl_version": v.value}

    def searchShardedHost(self, h_queries_ptr: int, nq: int, targetVectors: BinarizedByteVectorValues, k: int,
                          h_out_idx_ptr: int, h_out_score_ptr: int) -> int:
        """bbq_search_sharded on raw HOST pointers (pinned or pageable); returns the per-query result count."""
        self._one_gpu("searchShardedHost")
        cnt = C.c_uint32(0)
        _check(_native.load().bbq_search_sharded(_index(targetVectors), h_queries_ptr, nq, k, h_out_idx_ptr,
                                                 h_out_score_ptr, C.byref(cnt)), "search")
        return cnt.value

    def searchShardedDevice(self, d_queries_ptr: int, nq: int, targetVectors: BinarizedByteVectorValues, k: int,
                            d_out_idx_ptr: int, d_out_score_ptr: int, stream: int = 0):
        self._one_gpu("searchShardedDevice")
        _check(_native.load().bbq_search_sharded_device(_index(targetVectors), d_queries_ptr, nq, k, d_out_idx_ptr,
                                                        d_out_score_ptr, stream or None), "search")

    def mergeTopKDevice(self, d_idx_ptr: int, d_score_ptr: int, lists: int, nq: int, k: int, d_out_idx_ptr: int,
                        d_out_score_ptr: int, stream: int = 0):
        self._one_gpu("mergeTopKDevice")
        _check(_native.load().bbq_merge_topk_device(self._ctx, d_idx_ptr, d_score_ptr, lists, nq, k,
                                                    d_out_idx_ptr, d_out_score_ptr, stream or None), "search")

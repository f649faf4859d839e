"""A device group's index (GroupBinarizedByteVectorValues, a bbq_group_index* in C) never reaches a bbq_index_* entry:
every Python member that calls one refuses it with status 10 before any native call, and the one-GPU members refuse a
device-group format.  Needs no GPU: the objects are made without a device and the checks come first."""
import pytest

import bbq_b200
from bbq_b200 import BbqError, BinaryQuantizationFormat, GroupBinarizedByteVectorValues


@pytest.fixture
def group_index():
    gi = object.__new__(GroupBinarizedByteVectorValues)
    gi._h = None      # never dereferenced: the members below must refuse it first
    gi._n, gi._dim = 4, 8
    return gi


@pytest.fixture
def fmt():
    f = object.__new__(BinaryQuantizationFormat)
    f._group, f._ctx, f.config = None, None, {"queryBits": 4, "indexBits": 1}
    return f


def test_a_group_index_is_not_a_one_gpu_index():
    assert not issubclass(GroupBinarizedByteVectorValues, bbq_b200.BinarizedByteVectorValues)


def _members_taking_a_one_gpu_index(gi):
    q = [0.5] * 8
    return {
        "quantizeQueryVector": lambda f: f.quantizeQueryVector(q, gi),
        "appendRows": lambda f: f.appendRows(gi, rows=[q]),
        "writeIndexRows": lambda f: f.writeIndexRows(gi, "/nonexistent/x", 4),
        "writeIndexMeta": lambda f: f.writeIndexMeta(gi, "/nonexistent/x", 4, [0] * 5),
        "setBase": lambda f: f.setBase(gi, 0),
        "attachOriginalVectorsDevice": lambda f: f.attachOriginalVectorsDevice(gi, 0),
        "rerankOwnedDevice": lambda f: f.rerankOwnedDevice(gi, 0, 1, 0, 1, 0),
        "debugQcDist": lambda f: f.debugQcDist(q, gi),
        "debugQcDistBatch": lambda f: f.debugQcDistBatch([q], gi),
        "debugScores": lambda f: f.debugScores(q, gi),
        "searchDevice": lambda f: f.searchDevice(0, 1, gi, 1, 0, 0),
        "searchShardedHost": lambda f: f.searchShardedHost(0, 1, gi, 1, 0, 0),
        "searchShardedDevice": lambda f: f.searchShardedDevice(0, 1, gi, 1, 0, 0),
    }


def test_members_taking_a_one_gpu_index_refuse_a_group_index(fmt, group_index):
    for name, call in _members_taking_a_one_gpu_index(group_index).items():
        with pytest.raises(BbqError) as e:
            call(fmt)
        assert e.value.status == 10 and "device group" in str(e.value), name


def test_sharded_bootstrap_refuses_a_group_index(group_index):
    with pytest.raises(BbqError) as e:
        bbq_b200.ShardedSearcher(None, group_index, 0)
    assert e.value.status == 10


def test_one_gpu_members_refuse_a_group_format(fmt, group_index):
    fmt._group = object()   # a device-group format, as far as the checks can tell
    try:
        calls = dict(_members_taking_a_one_gpu_index(group_index))
        del calls["quantizeQueryVector"]   # runs on the group's first GPU
        calls.update({
            "quantizeVectorsDevice": lambda f: f.quantizeVectorsDevice(0, 1, 8),
            "accumulateCentroid": lambda f: f.accumulateCentroid(__import__("numpy").zeros(8, "float32"), 0, rows=[[0.0] * 8]),
            "reserveIndex": lambda f: f.reserveIndex(4, 8, [0.0] * 8),
            "loadIndexRows": lambda f: f.loadIndexRows("/nonexistent/x", 0, 1),
            "commInit": lambda f: f.commInit(b"\0" * 128, 0, 2),
            "commDestroy": lambda f: f.commDestroy(),
            "mergeTopKDevice": lambda f: f.mergeTopKDevice(0, 0, 1, 1, 1, 0, 0),
        })
        for name, call in calls.items():
            with pytest.raises(BbqError) as e:
                call(fmt)
            assert e.value.status == 10 and "device-group format" in str(e.value), name
    finally:
        fmt._group = None

"""Argument checks of the filtered searches that need no GPU: the C ABI rejects a NULL corpus, NULL ids with
n_filter > 0, an unknown mode and an oversized set before it touches a device, and the Python wrappers refuse
`within` together with `excluding`."""
import ctypes

import numpy as np
import pytest

from pixelbox_b200 import _native as nat
from pixelbox_b200.corpus import Corpus, MultiDeviceCorpus

PBX_MAX_ROWS = 0xFFFFF000


def _err():
    return nat.lib().pbx_last_error().decode()


def _host_calls(filter_ids, n_filter, mode):
    """The three host-form entry points with a NULL handle and valid buffers otherwise."""
    L = nat.lib()
    q = np.zeros((1, 8), np.uint8)
    ids, dist, dot, n2, cnt = np.zeros(10, np.int64), np.zeros(10, np.float32), np.zeros(10, np.int32), np.zeros(10, np.int32), np.zeros(1, np.uint32)
    hits = np.zeros(10, nat.HIT_DTYPE)
    fp = nat.ptr(filter_ids) if filter_ids is not None else None
    yield L.pbx_search_filtered(None, nat.ptr(q), 1, 10, 1e3, nat.ptr(ids), nat.ptr(dist), nat.ptr(dot), nat.ptr(n2), nat.ptr(cnt),
                                fp, n_filter, mode)
    yield L.pbx_sharded_search_filtered(None, nat.ptr(q), 1, 10, 1e3, nat.ptr(ids), nat.ptr(dist), nat.ptr(dot), nat.ptr(n2),
                                        nat.ptr(cnt), fp, n_filter, mode)
    yield L.pbx_exchange_search_hits_filtered(None, None, nat.ptr(q), 1, 10, 1e3, nat.ptr(hits), nat.ptr(cnt), fp, n_filter, mode)
    yield L.pbx_search_device_filtered(None, None, 1, 10, 1e3, None, None, None, fp, n_filter, mode)


def test_null_corpus_is_invalid():
    fids = np.array([3, 1, 2], np.int64)
    for rc in _host_calls(fids, 3, nat.PBX_FILTER_INCLUDE):
        assert rc == -1
        assert "NULL" in _err()


def test_null_ids_with_a_count_are_invalid():
    for rc in _host_calls(None, 5, nat.PBX_FILTER_INCLUDE):
        assert rc == -1 and "filter_ids is NULL" in _err()
    for rc in _host_calls(None, 1, nat.PBX_FILTER_EXCLUDE):
        assert rc == -1 and "filter_ids is NULL" in _err()


def test_unknown_mode_is_invalid():
    fids = np.array([1], np.int64)
    for mode in (2, 7, 0xFFFFFFFF):
        for rc in _host_calls(fids, 1, mode):
            assert rc == -1 and "unknown filter mode" in _err()


def test_oversized_set_is_invalid():
    fids = np.array([1], np.int64)          # never read: the size is rejected first
    for rc in _host_calls(fids, PBX_MAX_ROWS + 1, nat.PBX_FILTER_INCLUDE):
        assert rc == -1 and "PBX_MAX_ROWS" in _err()


def test_within_and_excluding_together_raise():
    with pytest.raises(ValueError):
        nat.filter_args([1, 2], [3])
    ids, mode = nat.filter_args(None, [4, 3])
    assert mode == nat.PBX_FILTER_EXCLUDE and ids.dtype == np.int64 and list(ids) == [4, 3]
    ids, mode = nat.filter_args([], None)
    assert mode == nat.PBX_FILTER_INCLUDE and ids.size == 0
    # the wrappers check before any native call: instances without a device handle are enough
    for cls in (Corpus, MultiDeviceCorpus):
        obj = cls.__new__(cls)
        obj._h, obj.dim = ctypes.c_void_p(0), 8
        with pytest.raises(ValueError):
            obj.search(np.zeros(8, np.uint8), 10, within=[1], excluding=[2])

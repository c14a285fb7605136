"""orbx_search_by_bow_batch without a device: the argument checks that run before any device work, n_kf == 0, and the C++
adapter driver of the two batched SearchByBoW overloads compiling and linking."""
import ctypes as C
import os

import numpy as np
import pytest

from tests import test_adapter_bow_batch_cpp
from wut_cuda_orb_slam3_b200 import capi
from wut_cuda_orb_slam3_b200.capi import BowViewC, FeatureVectorC, lib, ptr


def fv_arrays(nodes, offsets, indices):
    return (np.asarray(nodes, np.uint32), np.asarray(offsets, np.int32), np.asarray(indices, np.uint32))


class Case:
    """A fixed side of 4 features in nodes 1 and 2 and n_kf key frames of 3 features in nodes 2 and 5 (well-formed), with
    sentinel-filled outputs."""

    def __init__(self, n_kf):
        self.desc = np.arange(4 * 32, dtype=np.uint8).reshape(4, 32)
        self.angle = np.zeros(4, np.float32)
        self.valid = np.ones(4, np.uint8)
        self.fv = fv_arrays([1, 2], [0, 2, 4], [0, 1, 2, 3])
        self.kdesc = np.arange(3 * 32, dtype=np.uint8).reshape(3, 32)
        self.kangle = np.zeros(3, np.float32)
        self.kvalid = np.ones(3, np.uint8)
        self.kfv = fv_arrays([2, 5], [0, 1, 3], [0, 1, 2])
        self.views = (BowViewC * max(n_kf, 1))()
        for k in range(n_kf):
            self.set_view(k)
        self.n_kf = n_kf
        self.match = np.full(max(n_kf, 1) * 4, 12345, np.int32)
        self.nm = np.full(max(n_kf, 1), 777, np.int32)

    def set_view(self, k, fv=None, angle=True, valid=True, n=3):
        v = self.views[k]
        fv = fv if fv is not None else self.kfv
        self.__dict__.setdefault("keep", []).append(fv)
        v.n = n; v.desc = ptr(self.kdesc); v.angle = ptr(self.kangle) if angle else None; v.valid = ptr(self.kvalid) if valid else None
        v.fv = FeatureVectorC(len(fv[0]), ptr(fv[0]), ptr(fv[1]), ptr(fv[2]))

    def call(self, mode=0, nleft=-1, check_ori=1, n_kf=None, kfs=True, angle=True, valid=True, fv=None):
        fv = fv if fv is not None else self.fv
        f = FeatureVectorC(len(fv[0]), ptr(fv[0]), ptr(fv[1]), ptr(fv[2]))
        return lib().orbx_search_by_bow_batch(0, mode, ptr(self.desc), ptr(self.angle) if angle else None, ptr(self.valid) if valid else None,
                                              4, C.addressof(f), nleft, self.n_kf if n_kf is None else n_kf,
                                              C.addressof(self.views) if kfs else None, 0.75, check_ori, ptr(self.match), ptr(self.nm))

    def untouched(self):
        return (self.match == 12345).all() and (self.nm == 777).all()


def last_error():
    return lib().orbx_last_error().decode()


@pytest.mark.parametrize("mode", [0, 1])
def test_argument_errors_before_any_work(mode):
    c = Case(5)
    assert c.call(mode, n_kf=-1) == capi.ORBX_ERR_INVALID_ARG
    assert c.call(mode, kfs=False) == capi.ORBX_ERR_INVALID_ARG
    assert c.call(mode=2) == capi.ORBX_ERR_INVALID_ARG
    assert c.call(mode, n_kf=65536) == capi.ORBX_ERR_UNSUPPORTED
    # a malformed feature vector on a view that is not the first: node ids not ascending
    c.set_view(3, fv=fv_arrays([5, 2], [0, 1, 3], [0, 1, 2]))
    assert c.call(mode) == capi.ORBX_ERR_INVALID_ARG
    assert "kfs[3].fv" in last_error()
    # a feature index out of range on that view
    c.set_view(3, fv=fv_arrays([2, 5], [0, 1, 3], [0, 1, 3]))
    assert c.call(mode) == capi.ORBX_ERR_INVALID_ARG
    assert "kfs[3].fv" in last_error()
    # a malformed fixed feature vector
    c.set_view(3)
    assert c.call(mode, fv=fv_arrays([1, 2], [0, 3, 2], [0, 1, 2, 3])) == capi.ORBX_ERR_INVALID_ARG
    # NULL angles under check_orientation, on the fixed side and on a view
    assert c.call(mode, angle=False) == capi.ORBX_ERR_INVALID_ARG
    c.set_view(2, angle=False)
    assert c.call(mode) == capi.ORBX_ERR_INVALID_ARG
    assert "kfs[2]" in last_error()
    c.set_view(2)
    # NULL validity flags on a view (both modes read them), and a negative size
    c.set_view(4, valid=False)
    assert c.call(mode) == capi.ORBX_ERR_INVALID_ARG
    c.set_view(4, n=-1)
    assert c.call(mode) == capi.ORBX_ERR_INVALID_ARG
    assert c.untouched()


def test_mode_specific_errors():
    c = Case(2)
    # mode 1 (KF -> KF) takes no Nleft
    assert c.call(1, nleft=0) == capi.ORBX_ERR_INVALID_ARG
    assert c.call(1, nleft=3) == capi.ORBX_ERR_INVALID_ARG
    # mode 1 reads the fixed side's validity flags (KF1's map points)
    assert c.call(1, valid=False) == capi.ORBX_ERR_INVALID_ARG
    assert c.untouched()


@pytest.mark.parametrize("mode", [0, 1])
def test_no_key_frames_is_a_no_op(mode):
    c = Case(0)
    assert c.call(mode) == capi.ORBX_OK
    assert c.call(mode, kfs=False) == capi.ORBX_OK
    assert c.untouched()


def test_adapter_driver_compiles_and_links():
    """The two batched SearchByBoW overloads of csrc/adapter/ORBmatcher.h compile against the stand-ins and link with liborbx
    and the oracle."""
    test_adapter_bow_batch_cpp.build_exe()
    assert os.path.exists(test_adapter_bow_batch_cpp.EXE)

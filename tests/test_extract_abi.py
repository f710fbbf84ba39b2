"""CPU suite: argument validation of the volume-extraction entry points (inerf_volume_points, inerf_extract_volume) returns
its negative inerf_status before any launch, so none of these calls needs a GPU."""
import ctypes
import os

import numpy as np
import pytest

from instance_nerf_b200 import _lib

NULL_, SIZE, UNSUPPORTED = -1, -2, -3
FAKE = 0x10000   # a non-NULL "device" pointer: every call below is rejected before anything dereferences it


@pytest.fixture(scope="module")
def L():
    if not os.path.exists(_lib.LIB_PATH):
        _lib.build()
    return _lib.lib()


def _bbox(*v):
    return np.ascontiguousarray(v, dtype=np.float32)


def _desc(K=4, bound=8.0):
    d = _lib.FieldDesc()
    d.table_packed, d.offsets, d.weights = FAKE, FAKE, FAKE
    d.L, d.H, d.S, d.bound, d.K, d.density_scale = 16, 16, 1.0, bound, K, 1.0
    return d


GOOD = _bbox(-1, -1, -1, 1, 1, 1)
VD = _bbox(0, 0, 1)


def _points(L, bbox=GOOD, X=8, Y=8, Z=8, bits=None, C=4, H=128, bound=8.0, xyzs=FAKE, occ=None):
    return L.inerf_volume_points(None if bbox is None else bbox.ctypes.data, X, Y, Z, bits, C, H, bound, xyzs, occ, None)


def _extract(L, desc=None, bbox=GOOD, X=8, Y=8, Z=8, bits=None, C=4, H=128, vd=VD, sigma=FAKE, rgb=None, label=FAKE, scratch=FAKE):
    d = _desc() if desc is None else desc
    return L.inerf_extract_volume(ctypes.byref(d), None if bbox is None else bbox.ctypes.data, X, Y, Z, bits, C, H,
                                  None if vd is None else vd.ctypes.data, 0.5, sigma, rgb, label, scratch, None, None)


def test_version(L):
    assert L.inerf_version() == 1001


@pytest.mark.parametrize("X,Y,Z", [(0, 8, 8), (8, 0, 8), (8, 8, 0), (2049, 8, 8), (8, 2049, 8), (8, 8, 2049), (2048, 2048, 512)])
def test_bad_axes(L, X, Y, Z):
    # an axis of 0 or > 2048, or X * Y * Z >= 2^31 (2048 * 2048 * 512 = 2^31)
    assert _points(L, X=X, Y=Y, Z=Z) == SIZE
    assert _extract(L, X=X, Y=Y, Z=Z) == SIZE
    assert L.inerf_extract_scratch_ints(X, Y, Z) == 0


@pytest.mark.parametrize("bbox", [
    _bbox(-1, -1, -1, -1, 1, 1),      # hi == lo
    _bbox(-1, 2, -1, 1, 1, 1),        # hi < lo
    _bbox(-9, -1, -1, 1, 1, 1),       # outside [-bound, bound]
    _bbox(-1, -1, -1, 1, 1, 8.5),
    _bbox(-1, -1, -1, 1, float("nan"), 1),
])
def test_bad_bbox(L, bbox):
    assert _points(L, bbox=bbox) == SIZE
    assert _extract(L, bbox=bbox) == SIZE


def test_bbox_on_the_bound_is_accepted_up_to_the_launch(L):
    # the whole scene box is a valid request: everything is checked, then the call reaches the (absent) device
    full = _bbox(-8, -8, -8, 8, 8, 8)
    assert _points(L, bbox=full, xyzs=None) == NULL_


def test_null_pointers(L):
    assert _points(L, bbox=None) == NULL_
    assert _points(L, xyzs=None) == NULL_
    assert L.inerf_extract_volume(None, GOOD.ctypes.data, 8, 8, 8, None, 4, 128, None, 0.5, FAKE, None, None, None, None, None) == NULL_
    assert _extract(L, bbox=None) == NULL_
    d = _desc()
    d.weights = None
    assert _extract(L, desc=d) == NULL_
    # rgb needs the view direction; the occupancy pre-pass needs scratch
    assert _extract(L, rgb=FAKE, vd=None) == NULL_
    assert _extract(L, bits=FAKE, scratch=None) == NULL_


def test_no_outputs(L):
    assert _extract(L, sigma=None, rgb=None, label=None) == NULL_


def test_label_without_instances(L):
    assert _extract(L, desc=_desc(K=0)) < 0
    assert _extract(L, desc=_desc(K=0)) == UNSUPPORTED


def test_bad_occupancy_grid(L):
    for C, H in [(0, 128), (17, 128), (4, 100), (4, 1), (4, 2048)]:
        assert _points(L, bits=FAKE, C=C, H=H) == SIZE
        assert _extract(L, bits=FAKE, C=C, H=H) == SIZE


def test_bad_bound(L):
    assert _points(L, bound=0.0) == SIZE
    assert _extract(L, desc=_desc(bound=0.0)) == UNSUPPORTED   # the field descriptor is checked first


@pytest.mark.parametrize("X,Y,Z", [(1, 1, 1), (37, 20, 53), (256, 256, 256), (512, 512, 512), (2048, 2048, 511)])
def test_scratch_formula(L, X, Y, Z):
    # live ids (one per voxel, C order enumeration) | one count per 1024-voxel block of the pre-pass | the live count
    n = X * Y * Z
    assert L.inerf_extract_scratch_ints(X, Y, Z) == n + (n + 1023) // 1024 + 1

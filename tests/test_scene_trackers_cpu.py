"""Per-scene tracker table, host side: the ctypes mirror of mmw_scene_tracker against include/mmw.h, and the argument
handling of BatchedTracker.set_scene_trackers (against a stand-in for the library: no device needed)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from conftest import ROOT
from mmwave_msc_b200 import _lib
from mmwave_msc_b200.batched import BatchedTracker

_CTYPES = {"double": 8, "int32_t": 4, "float": 4}


def _header_struct(name):
    """(field, offset, size) of a plain C struct of include/mmw.h (scalars and fixed arrays, natural alignment)."""
    h = open(os.path.join(ROOT, "include", "mmw.h")).read()
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (name, name), h, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields, off, align = [], 0, 1
    for ctype, fname, n in re.findall(r"\b(double|int32_t|float)\s+(\w+)\s*(?:\[(\d+)\])?\s*;", body):
        al = _CTYPES[ctype]
        size = al * (int(n) if n else 1)
        off = (off + al - 1) // al * al
        fields.append((fname, off, size))
        off += size
        align = max(align, al)
    return fields, (off + align - 1) // align * align


def test_scene_tracker_layout_matches_header():
    fields, size = _header_struct("mmw_scene_tracker")
    got = [(f[0], getattr(_lib.SceneTracker, f[0]).offset, getattr(_lib.SceneTracker, f[0]).size)
           for f in _lib.SceneTracker._fields_]
    assert got == fields
    assert C.sizeof(_lib.SceneTracker) == size == 176
    assert [(n, _lib.SCENE_TRACKER_DTYPE.fields[n][1]) for n, _, _ in fields] == [(n, o) for n, o, _ in fields]
    assert _lib.SCENE_TRACKER_DTYPE.itemsize == size


def test_scene_tracker_fields_are_the_config_fields():
    """Same names as mmw_config; the context-wide ones (frames_batch, pose model, window geometry, sensor) are not in."""
    cfg = {f[0]: f[1] for f in _lib.Config._fields_}
    for name, ctype in _lib.SceneTracker._fields_:
        assert name in cfg and cfg[name] == ctype, name
    for name in ("frames_batch", "intensity_mu", "intensity_std", "default_posture", "m_x", "fade_weight", "s_height",
                 "doppler_res", "xyz_q_format"):
        assert name not in _lib.SCENE_TRACKER_DTYPE.names


class _FakeLib:
    """Stands in for libmmw.so: keeps a tracker table and records the tables handed to mmw_set_scene_trackers."""

    def __init__(self, S):
        self.table = np.zeros(S, _lib.SCENE_TRACKER_DTYPE)
        self.table["db_eps"] = 0.3
        self.table["db_min_samples"] = 35
        self.table["tr_max_tracks"] = 4
        self.table["kf_spread_lim"] = (0.2, 0.2, 2, 1.2, 1.2, 0.2)
        self.sets = []

    def mmw_get_scene_trackers(self, h, first, n, out):
        C.memmove(out.value, self.table.ctypes.data + first * self.table.itemsize, n * self.table.itemsize)
        return 0

    def mmw_set_scene_trackers(self, h, first, n, params):
        t = np.zeros(n, _lib.SCENE_TRACKER_DTYPE)
        C.memmove(t.ctypes.data, params.value, n * t.itemsize)
        self.sets.append((first, n))
        self.table[first:first + n] = t
        return 0


def _tracker(S=5):
    bt = object.__new__(BatchedTracker)
    bt.lib, bt._h, bt.S = _FakeLib(S), None, S
    return bt


def test_set_scene_trackers_scalars_arrays_and_selection():
    bt = _tracker()
    bt.set_scene_trackers(db_eps=0.45, tr_max_tracks=[10, 2], scenes=[1, 3])
    t = bt.lib.table
    np.testing.assert_array_equal(t["db_eps"], [0.3, 0.45, 0.3, 0.45, 0.3])
    np.testing.assert_array_equal(t["tr_max_tracks"], [4, 10, 4, 2, 4])
    assert bt.lib.sets == [(0, 5)]
    bt.set_scene_trackers(scenes=slice(3, None), kf_spread_lim=[0.1, 0.2, 0.3, 0.4, 0.5, 0.6])
    np.testing.assert_array_equal(t["kf_spread_lim"][3:], [[0.1, 0.2, 0.3, 0.4, 0.5, 0.6]] * 2)
    np.testing.assert_array_equal(t["kf_spread_lim"][0], [0.2, 0.2, 2, 1.2, 1.2, 0.2])
    per = np.arange(12, dtype=float).reshape(2, 6)
    bt.set_scene_trackers(scenes=[0, 4], kf_spread_lim=per)
    np.testing.assert_array_equal(t["kf_spread_lim"][[0, 4]], per)
    bt.set_scene_trackers(db_eps=None, db_min_samples=20.0)             # None keeps; an integral float is an integer
    np.testing.assert_array_equal(t["db_eps"], [0.3, 0.45, 0.3, 0.45, 0.3])
    assert np.all(t["db_min_samples"] == 20)
    assert bt.scene_trackers().tobytes() == t.tobytes()


@pytest.mark.parametrize("kw", [
    dict(db_min_samples=2.5), dict(tr_max_tracks=[1, 2.5, 3, 4, 5]), dict(kf_enable_est=0.5),
    dict(kf_est_pointnum=np.nan),
    dict(db_eps=[0.1, 0.2]), dict(db_eps=[[0.3] * 5]), dict(kf_spread_lim=[0.2] * 5),
    dict(kf_spread_lim=np.zeros((4, 6))), dict(kf_spread_lim=0.2), dict(no_such_field=1.0), dict(frames_batch=2),
])
def test_set_scene_trackers_refuses_bad_arguments_before_the_call(kw):
    bt = _tracker()
    before = bt.lib.table.copy()
    with pytest.raises((ValueError, AttributeError)):
        bt.set_scene_trackers(**kw)
    assert bt.lib.sets == [] and bt.lib.table.tobytes() == before.tobytes()

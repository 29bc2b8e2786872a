"""Per-scene sensor table, host side: the ctypes mirror of mmw_scene_sensor against include/mmw.h, and the synthetic
generator's mounting fields leaving the default scenes unchanged."""
import ctypes as C
import os
import re

import numpy as np

from conftest import GOLDEN, ROOT
from mmwave_msc_b200 import _lib, synth

_CTYPES = {"double": (8, 8), "int32_t": (4, 4), "float": (4, 4)}


def _header_struct(name):
    """(field, offset, size) of a plain C struct of include/mmw.h, laid out with natural alignment; and its size."""
    h = open(os.path.join(ROOT, "include", "mmw.h")).read()
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (name, name), h, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields, off, align = [], 0, 1
    for ctype, fname in re.findall(r"\b(double|int32_t|float)\s+(\w+)\s*;", body):
        size, al = _CTYPES[ctype]
        off = (off + al - 1) // al * al
        fields.append((fname, off, size))
        off += size
        align = max(align, al)
    return fields, (off + align - 1) // align * align


def test_scene_sensor_layout_matches_header():
    fields, size = _header_struct("mmw_scene_sensor")
    got = [(f[0], getattr(_lib.SceneSensor, f[0]).offset, getattr(_lib.SceneSensor, f[0]).size)
           for f in _lib.SceneSensor._fields_]
    assert got == fields
    assert C.sizeof(_lib.SceneSensor) == size == 40
    assert [(n, _lib.SCENE_SENSOR_DTYPE.fields[n][1]) for n, _, _ in fields] == [(n, o) for n, o, _ in fields]
    assert _lib.SCENE_SENSOR_DTYPE.itemsize == size


def test_default_spec_frames_are_unchanged():
    """The mounting fields of SceneSpec default to the module constants: scene 0 is still the golden trace's input."""
    g = np.load(os.path.join(GOLDEN, "c1_s0.npz"))
    sc = synth.gen_scene(0, 60)
    assert synth.SceneSpec().s_height == synth.S_HEIGHT and synth.SceneSpec().s_tilt_deg == synth.S_TILT_DEG
    assert np.array_equal(np.concatenate(sc.frames, axis=0), g["raw"])
    assert np.array_equal(np.cumsum([0] + [len(f) for f in sc.frames]), g["raw_off"])


def test_other_mounting_changes_the_sensor_frame_only():
    """A scene generated for another mounting is the same people seen from elsewhere: same point counts and peak
    values, other sensor-frame coordinates."""
    a = synth.gen_scene(3, 5)
    b = synth.gen_scene(3, 5, synth.SceneSpec(s_height=2.4, s_tilt_deg=-15.0))
    for fa, fb in zip(a.frames, b.frames):
        assert fa.shape == fb.shape
        np.testing.assert_array_equal(fa[:, 4], fb[:, 4])
        assert not np.array_equal(fa[:, 1:3], fb[:, 1:3])

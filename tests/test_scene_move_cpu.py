"""Host-side parts of the per-scene export / import: the scene-blob header and its parsing, and the argument checks of
sharding.move_scenes that need no device."""
import ctypes as C

import numpy as np
import pytest

from mmwave_msc_b200 import _lib
from mmwave_msc_b200.batched import scene_blob_info
from mmwave_msc_b200.sharding import move_scenes


def _blob(scenes, record_bytes=58960, ncap=256, tcap=8, fb=2, magic=_lib.SCENE_BLOB_MAGIC):
    n = len(scenes)
    head = 64 + (4 * n + 15) // 16 * 16
    total = head + n * record_bytes
    h = _lib.SceneBlobHeader(magic=magic, abi_version=_lib.ABI_VERSION, n=n, max_points_per_frame=ncap,
                             max_tracks=tcap, frames_batch=fb, record_bytes=record_bytes, total_bytes=total)
    out = np.zeros(total, np.uint8)
    out[:64] = np.frombuffer(bytes(h), np.uint8)
    out[64:64 + 4 * n] = np.asarray(scenes, np.int32).view(np.uint8)
    return out


def test_header_is_64_bytes_and_matches_the_c_header():
    import os
    import re
    from conftest import ROOT
    src = open(os.path.join(ROOT, "include", "mmw.h")).read()
    assert C.sizeof(_lib.SceneBlobHeader) == 64
    assert int(re.search(r"#define MMW_SCENE_BLOB_MAGIC (0x[0-9a-fA-F]+)", src).group(1), 16) == _lib.SCENE_BLOB_MAGIC
    body = re.search(r"typedef struct mmw_scene_blob_header \{(.*?)\} mmw_scene_blob_header;", src, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = re.findall(r"\b(\w+)(?:\[\d+\])?;", body)
    assert fields == [f for f, _ in _lib.SceneBlobHeader._fields_]


@pytest.mark.parametrize("scenes", [[], [5], [3, 7, 11], list(range(5)), list(range(1023, -1, -2))])
def test_scene_blob_info_reads_sizes_and_source_indices(scenes):
    b = _blob(scenes)
    info = scene_blob_info(b)
    assert info["n"] == len(scenes) and list(info["scenes"]) == scenes and info["scenes"].dtype == np.int32
    assert (info["max_points_per_frame"], info["max_tracks"], info["frames_batch"]) == (256, 8, 2)
    assert info["record_bytes"] == 58960 and info["total_bytes"] == b.size
    assert info["abi_version"] == _lib.ABI_VERSION
    assert b.size % 16 == 0
    # a blob inside a larger buffer (export_scenes with out=) parses the same
    assert list(scene_blob_info(np.concatenate([b, np.zeros(100, np.uint8)]))["scenes"]) == scenes


def test_scene_blob_info_rejects_bad_magic_and_truncation():
    b = _blob([1, 2, 3])
    with pytest.raises(ValueError, match="not a scene blob"):
        scene_blob_info(_blob([1, 2, 3], magic=0x4D4D5753))          # the whole-context blob's magic
    with pytest.raises(ValueError, match="truncated"):
        scene_blob_info(b[:-1])
    with pytest.raises(ValueError, match="truncated"):
        scene_blob_info(b[:40])
    bad = b.copy()
    bad[32:40] = np.array([64], np.uint64).view(np.uint8)            # total_bytes smaller than its records
    with pytest.raises(ValueError, match="inconsistent"):
        scene_blob_info(bad)


class _NoDevice:
    """Stands in for a BatchedTracker: any call into the library is a failure of the test."""

    def __getattr__(self, name):
        raise AssertionError("move_scenes touched the context (%s) before checking its arguments" % name)


def test_move_scenes_checks_arguments_first():
    a, b = _NoDevice(), _NoDevice()
    with pytest.raises(ValueError, match="destination"):
        move_scenes(a, [1, 2, 3], b, [0, 1])
    with pytest.raises(ValueError, match="same context"):
        move_scenes(a, [1, 2], a, [2, 5])

"""Dataset-builder mode of the reference's ``preprocessing.py`` (SURVEY 8(f) row 3) on the batched GPU path.

``preprocess_dataset`` of the reference (preprocessing.py:148-275) replays ONE recorded experiment at a time through
``normalize_data`` -> ``TrackBuffer.track`` and, for every frame in which track 0 was seen, exports the track's
three-frame point cloud (``relative_coordinates`` + ``format_batched_frames``) as CNN training input.  Here every
experiment is one scene of a ``BatchedTracker``: all experiments advance in lock step, one ``get_data()`` each per
device step, and ``mmw_export_track0`` produces the export blocks of all scenes at once.  The per-experiment control
flow (frame pairing, first-frame dt, ``batch.pop_frame()`` on missing frames, the invalid-frame list) is the
reference's, line for line.

Out of scope here, as in DESIGN.md: the Kinect side (``pair``, ``filter_kinect_frames``, ``kinect_z_correction``)
-- pass the paired mmWave frame numbers in ``frame_pairs``.
"""
from __future__ import annotations

import os
from dataclasses import dataclass, field
from typing import Dict, Iterable, List, Optional, Sequence

import numpy as np

from . import constants as const
from .Utils import OfflineManager, _doppler_units
from .batched import BatchedTracker, config_from_constants


@dataclass
class ExperimentExport:
    """What preprocess_dataset accumulates for one experiment."""
    name: str
    frames: List[int] = field(default_factory=list)            # frame numbers with a valid export ("Frame" column)
    rows: List[np.ndarray] = field(default_factory=list)       # (192, 5) float64 each: X, Y, Z, Doppler, Intensity
    centroids: List[np.ndarray] = field(default_factory=list)  # centroid[:2] per valid frame (preprocessing.py:209-213)
    invalid_frames: List[int] = field(default_factory=list)    # preprocessing.py:258-259

    def stacked(self):
        n = len(self.frames)
        return (np.asarray(self.frames, np.int64), np.stack(self.rows) if n else np.zeros((0, 192, 5)),
                np.stack(self.centroids) if n else np.zeros((0, 2)))


def _experiment_doppler_units(d: np.ndarray, own: Optional[float]):
    """``_doppler_units`` for one experiment: (index column, unit, own).  The unit in constants.DOPPLER_RESOLUTION (set,
    or found in an earlier experiment) is used while the experiment's values fit it; an experiment whose values do not
    (another radar profile) gets a unit of its own, ``own``, which it keeps."""
    shared = getattr(const, "DOPPLER_RESOLUTION", None)
    if own is None:
        try:
            idx, res = _doppler_units(d)
            return idx, res, None
        except ValueError:
            if shared is None:
                raise
    const.DOPPLER_RESOLUTION = None if own in (None, 1.0) else own
    try:
        idx, res = _doppler_units(d)
    finally:
        const.DOPPLER_RESOLUTION = shared
    return idx, res, res


def preprocess_dataset_batched(experiment_dirs: Sequence[str],
                               frame_pairs: Optional[Sequence[Optional[Iterable[int]]]] = None,
                               max_points: int = 256, max_tracks: int = 8, device: int = 0) -> List[ExperimentExport]:
    """Runs the frame loop of preprocess_dataset (preprocessing.py:167-259) for all experiments concurrently.

    experiment_dirs   directories with 1.csv, 2.csv, ... in the reference's log format (DataLogging.py:60-89)
    frame_pairs       per experiment the mmWave frame numbers that have a Kinect partner (``pair()[i][0]``,
                      preprocessing.py:175); None = every frame

    Every experiment keeps its own Doppler unit (experiments recorded with different radar profiles can share the
    run); the unit may not change within one experiment once it has shown a non-zero Doppler value.
    """
    E = len(experiment_dirs)
    if E == 0:
        return []
    pairs: List[Optional[set]] = [None] * E
    if frame_pairs is not None:
        if len(frame_pairs) != E:
            raise ValueError("frame_pairs must have one entry per experiment")
        pairs = [None if p is None else set(int(v) for v in p) for p in frame_pairs]
    readers = [OfflineManager(d) for d in experiment_dirs]
    out = [ExperimentExport(os.path.basename(os.path.normpath(d))) for d in experiment_dirs]
    bt = BatchedTracker(E, max_points=max_points, max_tracks=max_tracks, device=device,
                        config=config_from_constants(const))
    first_iter = [True] * E
    t_prev = [0.0] * E
    doppler_seen = False                 # a non-zero Doppler value has been stepped in any experiment
    seen = [False] * E                   # ... in this experiment
    unit = [bt.cfg.doppler_res] * E      # the Doppler unit of each scene on the device
    own = [None] * E                     # an experiment's own unit (see _experiment_doppler_units)
    per_scene = False                    # some scene has a unit of its own
    while True:
        live = [e for e in range(E) if not readers[e].is_finished()]
        if not live:
            break
        clouds = [np.zeros((0, 5), np.float32)] * E
        dts = np.full(E, 0.1)
        framenum = [None] * E
        stepped = [False] * E
        for e in live:
            data_ok, fn, det = readers[e].get_data()
            framenum[e] = fn
            if pairs[e] is not None and fn not in pairs[e]:
                continue
            if data_ok:
                if first_iter[e]:                                   # preprocessing.py:178-182
                    dts[e] = 0.1
                    first_iter[e] = False
                else:
                    dts[e] = det["posix"][0] / 1000 - t_prev[e]
                t_prev[e] = det["posix"][0] / 1000
                raw = np.stack([np.asarray(det[k], np.float64) for k in ("x", "y", "z", "doppler", "peakVal")], axis=1)
                raw32 = raw.astype(np.float32)
                if not np.array_equal(raw32[:, [0, 1, 2, 4]].astype(np.float64), raw[:, [0, 1, 2, 4]]):
                    raise ValueError("x, y, z, peakVal must be representable in float32 (int16/2^Q lattice values)")
                raw32[:, 3], res, own[e] = _experiment_doppler_units(raw[:, 3], own[e])   # the index; the device
                nonzero = bool(np.any(raw32[:, 3] != 0))                                # multiplies in float64
                if unit[e] != res and nonzero:                      # (zero rows are the same in every unit)
                    if seen[e]:
                        raise ValueError("Doppler resolution changes within experiment %s: set "
                                         "constants.DOPPLER_RESOLUTION" % out[e].name)
                    if not doppler_seen and not per_scene:
                        # nothing stepped so far has a non-zero Doppler value: the context's unit can change
                        bt.set_doppler_resolution(res)
                        unit = [res] * E
                    else:                                           # this experiment's radar profile differs
                        bt.set_scene_sensors(doppler_res=res, scenes=[e])
                        unit[e] = res
                        per_scene = True
                seen[e] = seen[e] or nonzero
                doppler_seen = doppler_seen or seen[e]
                clouds[e] = raw32
                stepped[e] = True
            else:
                bt.ring_pop(e)                                      # batch.pop_frame(), preprocessing.py:255-256
        if any(stepped):
            offsets = np.zeros(E + 1, np.int32)
            offsets[1:] = np.cumsum([len(c) for c in clouds])
            bt.step(np.concatenate(clouds, axis=0), offsets, dts, pose=False)
            rows, valid, cen = bt.export_track0()
        else:
            valid = np.zeros(E, bool)
        for e in live:
            if stepped[e] and valid[e]:                             # preprocessing.py:185-216
                out[e].frames.append(int(framenum[e]))
                out[e].rows.append(rows[e].copy())
                out[e].centroids.append(cen[e].copy())
            else:
                out[e].invalid_frames.append(int(framenum[e]))
    return out


def write_export_csv(export: ExperimentExport, output_dir: str) -> List[str]:
    """Writes one experiment the way preprocess_dataset does (preprocessing.py:218-262): rows
    ``Frame,X,Y,Z,Doppler,Intensity`` without header, 192 rows per frame, FB_EXPERIMENT_FILE_SIZE frames per n.csv."""
    import pandas as pd
    os.makedirs(output_dir, exist_ok=True)
    per_file = int(getattr(const, "FB_EXPERIMENT_FILE_SIZE", 200))
    paths = []
    for i in range(0, max(len(export.frames), 1), per_file):
        path = os.path.join(output_dir, "%d.csv" % (i // per_file + 1))
        chunks = []
        for fn, r in zip(export.frames[i:i + per_file], export.rows[i:i + per_file]):
            chunks.append(pd.DataFrame({"Frame": fn, "X": r[:, 0], "Y": r[:, 1], "Z": r[:, 2], "Doppler": r[:, 3],
                                        "Intensity": r[:, 4]}))
        (pd.concat(chunks, ignore_index=True) if chunks else pd.DataFrame()).to_csv(path, mode="w", index=False,
                                                                                   header=False)
        paths.append(path)
    return paths

"""TEST INFRASTRUCTURE ONLY -- pack/unpack per-frame trace records (the dicts
produced by ``ref_harness.run_reference_scene`` and ``mmw_oracle.SceneOracle.step``)
into flat arrays for ``tests/golden/*.npz``."""
from __future__ import annotations

import zipfile
from typing import Dict, List

import numpy as np

TRACK_VEC = {"x": 9, "P": 81, "spread_est": 6, "group_disp_est": 36, "centroid": 6, "min_vals": 6, "max_vals": 6}


def _pad3(a):
    out = np.full(3, -1, np.int32)
    a = np.asarray(a, np.int32)
    out[:len(a)] = a
    return out


def pack(frames: List[np.ndarray], dts: np.ndarray, recs: List[dict], feature_every: int = 7,
         doppler_res: float = 1.0, missing=None) -> Dict[str, np.ndarray]:
    """``frames``: fp32 rows as the device takes them -- Doppler column in units of ``doppler_res`` (the reference was
    run on row[3] * doppler_res in float64).  ``missing``: frames without sensor data (the global ring is popped)."""
    F = len(recs)
    d: Dict[str, np.ndarray] = {}
    d["doppler_res"] = np.array(doppler_res, np.float64)
    d["missing"] = np.zeros(F, bool) if missing is None else np.asarray(missing, bool)
    d["raw"] = np.concatenate(frames, axis=0).astype(np.float32)
    d["raw_off"] = np.cumsum([0] + [len(f) for f in frames]).astype(np.int64)
    d["dts"] = np.asarray(dts, np.float64)
    d["M"] = np.array([r["M"] for r in recs], np.int32)
    d["assoc"] = np.concatenate([np.asarray(r["assoc"], np.int16) for r in recs]) if F else np.zeros(0, np.int16)
    d["assoc_off"] = np.cumsum([0] + [len(r["assoc"]) for r in recs]).astype(np.int64)
    d["labels_ran"] = np.array([r["labels"] is not None for r in recs], bool)
    labs = [np.asarray(r["labels"], np.int16) if r["labels"] is not None else np.zeros(0, np.int16) for r in recs]
    d["labels"] = np.concatenate(labs) if F else np.zeros(0, np.int16)
    d["labels_off"] = np.cumsum([0] + [len(l) for l in labs]).astype(np.int64)
    d["ring_counts"] = np.stack([_pad3(r["ring_counts"][-3:]) for r in recs]) if F else np.zeros((0, 3), np.int32)
    d["next_track_id"] = np.array([r["next_track_id"] for r in recs], np.int32)
    d["ntracks"] = np.array([len(r["tracks"]) for r in recs], np.int32)
    tr = [t for r in recs for t in r["tracks"]]
    d["t_id"] = np.array([t["id"] for t in tr], np.int32)
    d["t_lifetime"] = np.array([t["lifetime"] for t in tr], np.float64)
    d["t_N_est"] = np.array([t["N_est"] for t in tr], np.float64)
    d["t_point_num"] = np.array([t["point_num"] for t in tr], np.int32)
    d["t_static"] = np.array([t["static"] for t in tr], bool)
    d["t_ring_counts"] = np.stack([_pad3(t["ring_counts"]) for t in tr]) if tr else np.zeros((0, 3), np.int32)
    for k, n in TRACK_VEC.items():
        d["t_" + k] = np.stack([np.asarray(t[k], np.float64).reshape(n) for t in tr]) if tr else np.zeros((0, n))
    sel = [f for f in range(F) if f % feature_every == 0 and recs[f].get("features") is not None]
    d["feat_frames"] = np.array(sel, np.int32)
    feats = [np.asarray(recs[f]["features"], np.float64) for f in sel]
    d["feat_off"] = np.cumsum([0] + [len(x) for x in feats]).astype(np.int64)
    d["feats"] = np.concatenate(feats, axis=0) if feats else np.zeros((0, 3, 8, 8, 5))
    return d


def save_npz(path: str, d: Dict[str, np.ndarray]) -> None:
    """``np.savez`` with LZMA instead of deflate (``np.load`` reads either): the float64 states of a long trace take
    about a seventh less room, which keeps every golden file under 1 MB."""
    with zipfile.ZipFile(path, "w", compression=zipfile.ZIP_LZMA) as z:
        for k, v in d.items():
            with z.open(k + ".npy", "w") as fh:
                np.lib.format.write_array(fh, np.asanyarray(v))


def unpack(d) -> dict:
    """Inverse of pack: returns {'frames', 'dts', 'recs'} with per-frame dicts."""
    F = len(d["M"])
    frames = [np.asarray(d["raw"][d["raw_off"][f]:d["raw_off"][f + 1]], np.float32) for f in range(F)]
    recs = []
    toff = np.cumsum([0] + list(d["ntracks"]))
    featmap = {int(f): k for k, f in enumerate(d["feat_frames"])}
    for f in range(F):
        r = {"M": int(d["M"][f]),
             "assoc": np.asarray(d["assoc"][d["assoc_off"][f]:d["assoc_off"][f + 1]], np.int32),
             "labels": (np.asarray(d["labels"][d["labels_off"][f]:d["labels_off"][f + 1]], np.int32)
                        if d["labels_ran"][f] else None),
             "ring_counts": np.asarray([c for c in d["ring_counts"][f] if c >= 0], np.int32),
             "next_track_id": int(d["next_track_id"][f]), "tracks": [], "features": None}
        for k in range(toff[f], toff[f + 1]):
            t = {"id": int(d["t_id"][k]), "lifetime": float(d["t_lifetime"][k]), "N_est": float(d["t_N_est"][k]),
                 "point_num": int(d["t_point_num"][k]), "static": bool(d["t_static"][k]),
                 "ring_counts": np.asarray([c for c in d["t_ring_counts"][k] if c >= 0], np.int32)}
            for name, n in TRACK_VEC.items():
                v = np.asarray(d["t_" + name][k], np.float64)
                t[name] = v.reshape(9, 9) if name == "P" else (v.reshape(6, 6) if name == "group_disp_est" else v)
            r["tracks"].append(t)
        if f in featmap:
            k = featmap[f]
            r["features"] = np.asarray(d["feats"][d["feat_off"][k]:d["feat_off"][k + 1]], np.float64)
        recs.append(r)
    files = getattr(d, "files", d)
    return {"frames": frames, "dts": np.asarray(d["dts"], np.float64), "recs": recs,
            "doppler_res": float(d["doppler_res"]) if "doppler_res" in files else 1.0,
            "missing": np.asarray(d["missing"], bool) if "missing" in files else np.zeros(F, bool)}


def reference_frames(g: dict) -> List[np.ndarray]:
    """The float64 rows the reference saw: Doppler column in m/s."""
    out = []
    for fr in g["frames"]:
        r = np.asarray(fr, np.float64).copy()
        r[:, 3] = r[:, 3] * g["doppler_res"]
        out.append(r)
    return out

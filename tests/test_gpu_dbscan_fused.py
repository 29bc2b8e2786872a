"""The DBSCAN kernels a tracker step runs (dbscan_big_kernel: the bit-matrix dbscan_bits_block for fused clouds of up
to min(3 max_points, 768) points, the pair-sweep dbscan_block<NbScreened> above that, both with the fp32 screen of the
eps predicate), held against the float64 oracle through BatchedTracker.step(record_labels=True): labels, spawned
tracks, ids and ring counts (helpers.compare_frame).

The clouds are built so that the kernels' edges decide the result: one pair straddling eps or the guard band decides
whether a cluster exists ((min_samples - 1) copies of A plus B), ties at d == eps, fused sizes across the 32-bit word
edges of the bit matrix, chains that need many frontier rounds, more than 32 clusters (the border step's row-pull
fallback), and the min_samples edges of the grid screen in front of the kernel.  Each scene holds one cloud;
reset_scenes starts every batch afresh."""
import numpy as np
import pytest

import dbscan_screen_model as sm
from helpers import compare_frame, oracle_config
from mmwave_msc_b200 import _lib
from mmwave_msc_b200.batched import BatchedTracker, default_config
from oracle import mmw_oracle as mo
from test_dbscan_screen_cpu import ISSUE_A, ISSUE_B
from test_grid_screen_cpu import screen_may_have_core

pytestmark = pytest.mark.gpu

DT = 0.1


def _bits_cap(ncap):
    return min(3 * ncap, 768)


def _tracker(ncap, n_scenes, tcap=8, **cfg):
    c = default_config(**cfg)
    return BatchedTracker(n_scenes, max_points=ncap, max_tracks=tcap, config=c), oracle_config(c)


def _oracle_rows(rows, rep):
    """float64 rows the oracle sees: dequantized int16 rows (doppler index 0), or the fp32 values."""
    out = np.asarray(rows, np.float64).copy()
    if rep is not None:
        out[:, :3] /= 2.0 ** rep
    return out


def _run(bt, ocfgs, frames, ctx, mounts=None, reps=None, check=True):
    """frames: per step, one (rows, rep) or None per scene (all rows of a step fp32, or all int16).  Resets the scenes,
    sets their mounting and Q format, steps, compares every frame with the oracle; returns the last records."""
    S = bt.S
    bt.reset_scenes(slice(None))
    mounts = mounts or [sm.MOUNTS[0]] * S
    qf = [9 if r is None else r for r in (reps or [None] * S)]
    bt.set_scene_sensors(s_height=[m.s_height for m in mounts], s_tilt_deg=[m.s_tilt_deg for m in mounts],
                         z_max=[m.z_max for m in mounts], xyz_q_format=qf)
    oracles = []
    for s in range(S):
        oc = mo.OracleConfig(**{k: getattr(ocfgs, k) for k in ocfgs.__dataclass_fields__})
        oc.s_height, oc.s_tilt_deg, oc.z_max = mounts[s].s_height, mounts[s].s_tilt_deg, mounts[s].z_max
        oracles.append(mo.SceneOracle(oc))
    recs = None
    for f, per in enumerate(frames):
        i16 = any(p is not None and p[0].dtype == np.int16 for p in per)
        dtype = np.int16 if i16 else np.float32
        parts = [np.zeros((0, 5), dtype) if p is None else p[0] for p in per]
        off = np.zeros(S + 1, np.int32)
        off[1:] = np.cumsum([len(p) for p in parts])
        bt.step(np.ascontiguousarray(np.concatenate(parts, 0)), off, np.full(S, DT), pose=False, record_labels=True)
        recs = [o.step(_oracle_rows(parts[s], None if p is None or p[0].dtype != np.int16 else p[1]), DT)
                for s, (o, p) in enumerate(zip(oracles, per))]
        if check:
            compare_frame(bt, recs, off, "%s step %d" % (ctx, f), labels=bt.labels())
    return recs


def _deferred(world, ocfg):
    """The step kernel hands the scene to dbscan_big_kernel: enough points, and a point beyond the grid screen's
    range bound or a block of cells that may hold a core point."""
    return len(world) >= ocfg.db_min_samples and (
        np.any(world[:, 1] > 12.0) or screen_may_have_core(world, ocfg))


def _decisive(p: sm.Pair, labels):
    """One pair decides: with it the (min_samples - 1) copies of A and B form one cluster, without it all are noise."""
    lab = np.asarray(labels)
    if p.neighbours():
        assert np.all(lab == 0), (p.family, p.target, lab)
    else:
        assert np.all(lab == -1), (p.family, p.target, lab)


def _pairs_for(cfg: sm.Cfg, rng):
    pairs = [p for p in sm.adversarial_pairs([cfg]) if p.rep != 10 or p.family in ("near_x", "near_y")]
    if cfg.rw > 0:
        for m in sm.MOUNTS:
            for rep in (None, 8, 9):
                pairs += sm.w0_search(cfg, m, rep, 200, rng)
    if cfg.name == "default":
        pairs.append(sm.Pair("issue", cfg, sm.MOUNTS[0], 9, ISSUE_A, ISSUE_B, "eps_below"))
    return pairs


def _pad_noise(rep, m: sm.Mount, n=820):
    """Points pairwise out of reach (1.2 m grid over 1 < y' < 25, so w >= 0.28 at the default range weight) and far
    from the w -> 0 pairs (mean y' 33 m), raw rows in the representation."""
    xs = np.arange(-24.0, 24.01, 1.2)
    ys = 1.0 + 1.2 * np.arange(20)
    pts = np.array([[x, y, 1.0] for y in ys for x in xs])[:n]
    raw = np.stack([sm.quantize(sm.to_raw(p, m), rep) for p in pts])
    if rep is None:
        out = np.zeros((len(raw), 5), np.float32)
        out[:, :3] = raw
    else:
        out = np.zeros((len(raw), 5), np.int16)
        out[:, :3] = np.rint(raw * 2.0 ** rep)
    out[:, 4] = 100
    return out


def _batches(items, S):
    for k in range(0, len(items), S):
        yield items[k:k + S]


# ---- 1. guard band, bit-matrix path -------------------------------------------------------------------------------
@pytest.mark.parametrize("cfg", sm.CONFIGS, ids=[c.name for c in sm.CONFIGS])
def test_guard_band_bit_matrix(cfg):
    rng = np.random.default_rng(7)
    pairs = _pairs_for(cfg, rng)
    ms = 35
    S = 256
    bt, ocfg = _tracker(256, S, db_eps=cfg.eps, db_range_weight=cfg.rw, db_z_weight=cfg.zw)
    for i16 in (False, True):
        sel = [p for p in pairs if (p.rep is not None) == i16]
        assert sel
        for batch in _batches(sel, S):
            frames = [[(p.rows(ms - 1), p.rep) for p in batch] + [None] * (S - len(batch))]
            mounts = [p.mount for p in batch] + [sm.MOUNTS[0]] * (S - len(batch))
            reps = [p.rep for p in batch] + [None] * (S - len(batch))
            recs = _run(bt, ocfg, frames, "%s i16=%d" % (cfg.name, i16), mounts, reps)
            for p, r in zip(batch, recs):
                w = r["world"][:, :3]
                assert len(w) == ms and _deferred(w, ocfg) and ms <= _bits_cap(256)
                _decisive(p, r["labels"])
    bt.close()


# ---- 2. guard band, pair-sweep path (A and B in different ring frames) ------------------------------------------------
def test_guard_band_pair_sweep():
    cfg = sm.CONFIGS[0]
    rng = np.random.default_rng(8)
    # the families whose A and B lie beyond y' = 25 m, clear of the padding
    pairs = [p for p in _pairs_for(cfg, rng) if p.family in ("w0_dx", "wneg", "w0_search", "issue")]
    assert any(p.family == "issue" for p in pairs) and any(p.family == "w0_search" for p in pairs)
    ms, S = 35, 64
    bt, ocfg = _tracker(1024, S)
    for i16 in (False, True):
        sel = [p for p in pairs if (p.rep is not None) == i16]
        for batch in _batches(sel, S):
            f0, f1 = [], []
            for p in batch:
                a = p.rows(ms - 1)
                noise = _pad_noise(p.rep, p.mount)
                f0.append((np.concatenate([a[:-1], noise]).astype(a.dtype), p.rep))   # A copies + noise
                f1.append((a[-1:], p.rep))                                           # B, one step later
            pad = S - len(batch)
            mounts = [p.mount for p in batch] + [sm.MOUNTS[0]] * pad
            reps = [p.rep for p in batch] + [None] * pad
            recs = _run(bt, ocfg, [f0 + [None] * pad, f1 + [None] * pad], "sweep i16=%d" % i16, mounts, reps)
            for p, r in zip(batch, recs):
                w = r["world"]
                B = len(r["labels"])
                assert B > _bits_cap(1024) and B >= ms and np.any(w[:, 1] > 12.0)
                lab = np.asarray(r["labels"])
                _decisive(p, np.concatenate([lab[:ms - 1], lab[-1:]]))
                assert np.all(lab[ms - 1:-1] == -1)
    bt.close()


# ---- 3. exact ties d == eps ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("ncap", [256, 1024], ids=["bits", "sweep"])
def test_exact_ties(ncap):
    m = sm.Mount("level", s_height=1.8, s_tilt_deg=0.0, z_max=2.5)
    ms, S = 35, 8
    bt, ocfg = _tracker(ncap, S, s_tilt_deg=0.0, db_range_weight=0.0, db_z_weight=0.0, db_eps=0.25)
    cases = []
    for rep in (None, 8, 9, 10):
        h = 2.0 ** -rep if rep is not None else float(np.spacing(np.float32(1.5)))
        for dx, want in ((0.5, True), (0.5 + h, False)):
            a = np.array([1.0, 28.0, -0.5])
            b = a + np.array([dx, 0.0, 0.3])                       # dz does not count (z weight 0)
            cases.append((sm.Pair("tie", sm.Cfg("tie", 0.25, 0.0, 0.0), m, rep, a, b, "tie"), want))
    frames = [[], []]
    for p, want in cases:
        assert p.neighbours() == want and (p.d() == 0.25) == want
        rows = p.rows(ms - 1)
        if ncap == 1024:
            noise = _pad_noise(p.rep, m)
            frames[0].append((np.concatenate([rows[:-1], noise]).astype(rows.dtype), p.rep))
            frames[1].append((rows[-1:], p.rep))
        else:
            frames[0].append((rows, p.rep))
    for i16 in (False, True):
        idx = [k for k, (p, _) in enumerate(cases) if (p.rep is not None) == i16]
        fr = [[f[k] for k in idx] + [None] * (S - len(idx)) for f in frames if f]
        reps = [cases[k][0].rep for k in idx] + [None] * (S - len(idx))
        recs = _run(bt, ocfg, fr, "ties %s i16=%d" % (ncap, i16), [m] * S, reps)
        for k, r in zip(idx, recs):
            lab = np.asarray(r["labels"])
            assert (len(lab) > _bits_cap(ncap)) == (ncap == 1024)
            _decisive(cases[k][0], np.concatenate([lab[:ms - 1], lab[-1:]]))
    bt.close()


# ---- 4. bit-matrix structure ----------------------------------------------------------------------------------------
def _cloud(world_pts):
    raw = np.stack([sm.to_raw(p, sm.MOUNTS[0]) for p in world_pts]).astype(np.float32)
    out = np.zeros((len(raw), 5), np.float32)
    out[:, :3] = raw
    out[:, 4] = 100
    return out


def test_bit_matrix_structure():
    rng = np.random.default_rng(11)
    ms = 5
    clouds = []
    for n in (1, 31, 32, 33, 63, 64, 65, 97, 255, 256, 257, 511, 767, 768, 769):
        L = 0.33 * np.sqrt(n)
        clouds.append(("random %d" % n, np.stack([rng.uniform(-L, L, n), rng.uniform(1.0, 1.0 + 2 * L, n),
                                                  rng.uniform(0.2, 2.2, n)], 1)))
        blobs = rng.uniform([-8, 2, 0.5], [8, 10, 2.0], (max(1, n // 40), 3))
        k = rng.integers(0, len(blobs), n)
        clouds.append(("blobs %d" % n, blobs[k] + rng.normal(0, 0.15, (n, 3)) * [1, 1, 0.3]))
    clouds.append(("identical 700", np.tile([[0.5, 3.0, 1.0]], (700, 1))))
    step = 0.999 * np.sqrt(0.3 / (1 - 0.03 * 3.0))               # just inside reach at y' = 3
    clouds.append(("chain 700", np.stack([np.arange(700) * step / 20 - 8, 3.0 + np.zeros(700), np.ones(700)], 1)))
    x = np.repeat(np.arange(80) * step - 12, 2)                 # two points per link: 6 neighbours, core
    clouds.append(("long chain", np.stack([x, 3.0 + np.zeros(160), np.ones(160)], 1)))
    # two tight clusters and border points within reach of both (the lower cluster id wins)
    sq = np.array([[0, 0, 0], [0.3, 0, 0], [0, 0.3, 0], [0.3, 0.3, 0], [0.15, 0.15, 0]])
    two = np.concatenate([sq + [1.04, 2.0, 1.0], sq + [-0.3, 2.0, 1.0], [[0.52, 2.0, 1.0], [0.52, 2.05, 1.0]]])
    clouds.append(("border of two", two))
    clouds.append(("border of two, swapped", np.concatenate([two[5:10], two[:5], two[10:]])))
    S = len(clouds)
    bt, ocfg = _tracker(1024, S, db_min_samples=ms, tr_max_tracks=64, tcap=32)
    frames = [[(_cloud(c), None) for _, c in clouds]]
    recs = _run(bt, ocfg, frames, "structure", check=False)
    lab, nf = bt.labels()
    st = bt.status()
    for s, ((name, _), r) in enumerate(zip(clouds, recs)):
        if r["labels"] is None:
            assert nf[s] == -1, name
            continue
        assert nf[s] == len(r["labels"]), name
        np.testing.assert_array_equal(lab[s, :nf[s]], r["labels"], err_msg=name)
        ncl = int(np.max(r["labels"], initial=-1)) + 1
        if ncl <= 32:
            assert not st[s] & _lib.SCENE_TRACK_OVERFLOW, name
    byname = {name: r for (name, _), r in zip(clouds, recs)}
    assert np.all(np.asarray(byname["identical 700"]["labels"]) == 0)
    assert np.all(np.asarray(byname["chain 700"]["labels"]) == 0)
    assert np.all(np.asarray(byname["long chain"]["labels"]) == 0)
    for nm in ("border of two", "border of two, swapped"):
        l2 = np.asarray(byname[nm]["labels"])
        assert set(l2[:10]) == {0, 1} and np.all(l2[10:] == 0), (nm, l2)
    bt.close()


# ---- 5. more than 32 clusters ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_clusters", [30, 46], ids=["masks", "row_pull"])
def test_many_clusters(n_clusters):
    """Clusters are 2 x 2 squares (side 0.3 m) on two rows; a border point between horizontal neighbours reaches one
    corner of each.  The squares are listed in a shuffled order, so neighbouring clusters get ids on both sides of 32."""
    ms = 4
    rng = np.random.default_rng(n_clusters)
    cols = (n_clusters + 1) // 2
    sq = np.array([[0, 0, 0], [0.3, 0, 0], [0, 0.3, 0], [0.3, 0.3, 0]])
    origin = [(-15.0 + 1.34 * (k % cols), 2.0 + 1.5 * (k // cols), 1.0) for k in range(n_clusters)]
    order = rng.permutation(n_clusters)
    pts = [sq + origin[k] for k in order]
    border = [(origin[k][0] + 0.3 + 0.52, origin[k][1], 1.0) for k in range(n_clusters) if (k + 1) % cols]
    cloud = np.concatenate(pts + [np.array(border)])
    bt, ocfg = _tracker(1024, 2, db_min_samples=ms, tr_max_tracks=64, tcap=32)
    w = sm.world(sm.to_raw(cloud.T, sm.MOUNTS[0]).T.astype(np.float32))
    want = mo.dbscan_labels(np.concatenate([w, np.zeros((len(w), 5))], 1), ocfg)
    assert want.max() + 1 == n_clusters
    nb = want[len(pts) * 4:]
    assert np.all(nb >= 0)                                       # every border point joined a cluster
    adj = mo.pair_distance_matrix(w, ocfg) <= ocfg.db_eps
    core = adj.sum(1) >= ms
    reach = [sorted(set(want[adj[i] & core])) for i in range(len(pts) * 4, len(w))]
    assert all(len(r) == 2 and want[len(pts) * 4 + i] == r[0] for i, r in enumerate(reach))
    if n_clusters > 32:
        assert any(r[0] < 32 <= r[1] for r in reach) and any(r[0] >= 32 for r in reach)
    frames = [[(_cloud(cloud), None), None]]
    recs = _run(bt, ocfg, frames, "clusters %d" % n_clusters, check=n_clusters <= 32)
    lab, nf = bt.labels()
    np.testing.assert_array_equal(lab[0, :nf[0]], want)
    np.testing.assert_array_equal(recs[0]["labels"], want)
    assert bool(bt.status()[0] & _lib.SCENE_TRACK_OVERFLOW) == (n_clusters > 32)
    assert len(want) <= _bits_cap(1024)
    bt.close()


# ---- 6. min_samples edges -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ms", [1, 2, 35, 255, 256])
def test_min_samples_edges(ms):
    bt, ocfg = _tracker(256, 4, db_min_samples=ms)
    rng = np.random.default_rng(ms)
    blob = lambda n: np.array([0.2, 3.0, 1.0]) + rng.normal(0, 0.05, (n, 3))     # noqa: E731
    frames = [[(_cloud(blob(ms - 1)), None) if ms > 1 else None, (_cloud(blob(ms)), None),
               (_cloud(np.tile([[0.2, 3.0, 1.0]], (ms, 1))), None), (_cloud(blob(ms - 1) + [0, 20, 0]), None)
               if ms > 1 else None]]
    recs = _run(bt, ocfg, frames, "min_samples %d" % ms)
    assert recs[1]["labels"] is not None and np.all(np.asarray(recs[1]["labels"]) == 0)
    assert np.all(np.asarray(recs[2]["labels"]) == 0)
    if ms > 1:
        assert np.all(np.asarray(recs[0]["labels"]) == -1) and np.all(np.asarray(recs[3]["labels"]) == -1)
    bt.close()

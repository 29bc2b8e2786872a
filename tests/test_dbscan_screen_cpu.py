"""The fp32 screen of DBSCAN's eps predicate (csrc/dbscan.cuh: screen_d, screen_domain_mark, screen_config), through
its numpy restatement in dbscan_screen_model.py: no fp32 decision may differ from the float64 predicate's -- on pairs
constructed to straddle eps and the edges of the guard band, on pairs where the range weight w vanishes or turns
negative, and on a seeded sweep of the admitted domain -- under both contraction extremes.  The rule without the domain
(the guard band alone) must fail on the w -> 0 pairs, so that these tests can tell the two apart."""
import numpy as np
import pytest

import dbscan_screen_model as sm

# Two raw rows on the Q9 lattice, 104 m apart, mean y' 33.33 m (w ~ 3e-5 at the default range weight 0.03): the float64
# distance is 0.2999617 <= eps, the fp32 distance 0.30074 (each operation rounded) or 0.30047 (contracted), above hi.
ISSUE_A = np.array([-54.4609375, 33.404296875, 1.46484375])
ISSUE_B = np.array([49.369140625, 33.158203125, 2.615234375])


def _check(wa, wb, cfg, band_only=False):
    """Number of pairs whose decision differs from the float64 predicate's, per contraction."""
    ex = sm.exact_d(wa, wb, cfg.rw, cfg.zw) <= cfg.eps
    return [int((sm.decisions(wa, wb, cfg.eps, cfg.rw, cfg.zw, f, band_only) != ex).sum()) for f in (False, True)]


@pytest.fixture(scope="module")
def pairs():
    return sm.adversarial_pairs()


@pytest.fixture(scope="module")
def w0_pairs():
    rng = np.random.default_rng(20261021)
    out = []
    for cfg in sm.CONFIGS:
        if cfg.rw > 0:
            for m in sm.MOUNTS:
                for rep in sm.REPS:
                    out += sm.w0_search(cfg, m, rep, 400, rng)
    return out


def test_issue_pair_needs_the_domain():
    wa, wb = sm.world(ISSUE_A), sm.world(ISSUE_B)
    cfg = sm.CONFIGS[0]
    assert sm.in_scene(wa).all() and sm.in_scene(wb).all()
    assert sm.exact_d(wa, wb, cfg.rw, cfg.zw)[0] <= cfg.eps
    lo, hi, rmax = sm.screen_config(cfg.eps, cfg.rw, cfg.zw)
    for fma in (False, True):
        d = sm.screen_d(wa.astype(np.float32), wb.astype(np.float32), cfg.rw, cfg.zw, fma)[0]
        assert d > hi, (fma, d, hi)                              # the band alone says "not neighbours"
    assert _check(wa, wb, cfg, band_only=True) == [1, 1]
    assert _check(wa, wb, cfg) == [0, 0]
    assert wa[0, 1] > rmax and wb[0, 1] > rmax                   # both outside the domain: decided in float64


def test_constructed_pairs_straddle_their_targets(pairs):
    fams = {p.family for p in pairs}
    assert {"near_x", "near_y", "y20_x", "y20_y", "w0_dx", "w0_dy", "wneg", "far_dy"} <= fams, fams
    for rep in sm.REPS:
        assert any(p.rep == rep for p in pairs), rep
    by = {}
    for p in pairs:
        by.setdefault((p.family, p.cfg.name, p.mount.name, p.rep, p.target[:-6]), []).append(p)
    for k, v in by.items():
        if k[4] == "eps":                                        # the pair just below eps and the pair just above
            assert sorted(p.neighbours() for p in v) == [False, True], k
    wneg = [p for p in pairs if p.family == "wneg"]
    assert wneg and all(p.d() <= 0 for p in wneg)


def test_no_decision_differs_on_constructed_pairs(pairs):
    for p in pairs:
        wa, wb = p.worlds()
        assert _check(wa[None], wb[None], p.cfg) == [0, 0], (p.family, p.cfg, p.mount.name, p.rep, p.target)


def test_band_alone_fails_where_w_vanishes(w0_pairs):
    assert len(w0_pairs) >= 10
    assert any(p.neighbours() for p in w0_pairs)
    assert {p.rep for p in w0_pairs} >= {None, 8}
    for p in w0_pairs:
        wa, wb = p.worlds()
        assert sum(_check(wa[None], wb[None], p.cfg, band_only=True)) > 0
        assert _check(wa[None], wb[None], p.cfg) == [0, 0], (p.cfg, p.mount.name, p.rep, p.a, p.b)


@pytest.mark.parametrize("cfg", sm.CONFIGS, ids=[c.name for c in sm.CONFIGS])
@pytest.mark.parametrize("mount", sm.MOUNTS, ids=[m.name for m in sm.MOUNTS])
@pytest.mark.parametrize("rep", sm.REPS, ids=["fp32", "q8", "q9", "q10"])
def test_random_sweep_of_the_domain(cfg, mount, rep):
    rng = np.random.default_rng([int(1e3 * cfg.eps), int(1e3 * cfg.rw), len(mount.name), rep or 0])
    wa, wb = sm.random_domain(60000, rng, cfg, mount, rep)
    assert len(wa) > 10000
    assert _check(wa, wb, cfg) == [0, 0]
    # the derivation's bound holds wherever the fp32 decision is taken
    lo, hi, rmax = sm.screen_config(cfg.eps, cfg.rw, cfg.zw)
    fa, fb = sm.screen_coords(wa, rmax), sm.screen_coords(wb, rmax)
    inside = np.isfinite(fa[:, 0]) & np.isfinite(fb[:, 0])
    assert inside.sum() > 1000
    d = sm.exact_d(wa, wb, cfg.rw, cfg.zw)[inside]
    w = 1.0 - ((wa[:, 1] + wb[:, 1]) * 0.5)[inside] * cfg.rw
    bound = sm.error_bound(d / w, rmax, cfg.zw)
    for fma in (False, True):
        err = np.abs(sm.screen_d(fa[inside], fb[inside], cfg.rw, cfg.zw, fma).astype(np.float64) - d)
        assert np.all(err <= bound), float((err / bound).max())


def test_screen_config_domain():
    eps = 0.3
    _, _, r = sm.screen_config(eps, 0.03, 0.4)
    assert r == np.float32(25.0)                                 # w >= 0.25 over the domain
    _, _, r0 = sm.screen_config(eps, 0.0, 0.4)
    assert 100 < r0 < 1000                                       # range weight 0: the input rounding of y' bounds it
    for bad in ((0.0, 0.03, 0.4), (-1.0, 0.03, 0.4), (eps, -0.01, 0.4), (eps, 0.03, -0.1), (np.nan, 0.03, 0.4),
                (eps, np.inf, 0.4), (eps, 0.03, np.nan)):
        assert sm.screen_config(*bad)[2] == -1, bad             # every pair decided in float64
    wa, wb = sm.world(ISSUE_A), sm.world(ISSUE_B)
    assert (sm.screened(wa, wb, eps, -0.01, 0.4) == -1).all()

"""The fp32 screen of DBSCAN's eps predicate in the tracker step (mmwave_msc_b200/csrc/dbscan.cuh: screen_d,
screen_domain_mark, screen_config; the float64 predicate is eps_neighbour in mmw_internal.cuh), restated in numpy, and
constructors of adversarial point pairs for it.

The kernels keep the world coordinates of the fused ring in fp32 (x as given, y' and z' rounded from the float64
transform), compute the weighted distance in fp32 and decide a pair from that alone when it is above hi or below lo;
everything else -- the guard band, and every pair with a point outside the screen's domain |y'|, |z'| <= rmax (its x
is NaN) -- is decided by the float64 predicate.  ``screened`` restates that with the fp32 arithmetic evaluated two ways:
every operation rounded on its own, and with the multiply-adds the compiler may contract fused.

``band_only=True`` drops the domain (the rule before it existed): a pair is decided in fp32 whenever its fp32 distance is
outside the band."""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import List, Optional, Tuple

import numpy as np

F32 = np.float32
U = 2.0 ** -24


# ---- the arithmetic of the kernels ----------------------------------------------------------------------------------
def world(raw, s_height=1.8, s_tilt_deg=-5.0) -> np.ndarray:
    """(n, 3) raw sensor rows (float64 values, after dequantization) -> float64 world (x, y', z') as world_yz computes
    them (and the oracle's normalize_points)."""
    raw = np.asarray(raw, np.float64).reshape(-1, 3)
    ang = np.radians(s_tilt_deg)
    c, s = np.cos(ang), np.sin(ang)
    x, y, z = raw[:, 0], raw[:, 1], raw[:, 2]
    return np.stack([x, c * y + (-s) * z, (s * y + c * z) + s_height], axis=1)


def in_scene(w, z_max=2.5) -> np.ndarray:
    """The scene filter of normalize_data (Utils.py:423-427)."""
    w = np.asarray(w, np.float64).reshape(-1, 3)
    return (w[:, 2] <= z_max) & (w[:, 2] > 0) & (w[:, 1] > 0)


def exact_d(a, b, rw, zw) -> np.ndarray:
    """eps_neighbour's float64 distance, operation for operation."""
    a = np.asarray(a, np.float64).reshape(-1, 3)
    b = np.asarray(b, np.float64).reshape(-1, 3)
    w = 1.0 - ((a[:, 1] + b[:, 1]) * 0.5) * rw
    dx, dy, dz = a[:, 0] - b[:, 0], a[:, 1] - b[:, 1], a[:, 2] - b[:, 2]
    return w * ((dx * dx + dy * dy) + zw * (dz * dz))


def screen_config(eps, rw, zw) -> Tuple[np.float32, np.float32, np.float32]:
    """screen_config: (lo, hi, rmax), fp32 like the host code.  rmax = -1: every pair is decided in float64."""
    band = F32(1e-3) * F32(eps) + F32(1e-4)
    lo, hi = F32(eps) - band, F32(eps) + band
    if not (0 < eps < 1e30 and 0 <= rw < 1e30 and 0 <= zw < 1e30):
        return lo, hi, F32(-1)
    wmin = 0.25
    Q = 2.0 * (eps + float(band)) / wmin
    R = (0.5 * float(band) - 22.0 * U * Q) / (8.0 * U * math.sqrt(Q) * (1.0 + math.sqrt(zw)))
    if rw > 0:
        R = min(R, (1.0 - wmin) / rw)
    if not R > 0:
        return lo, hi, F32(-1)
    R = min(R, 1e30)
    r = F32(R)
    if float(r) > R:
        r = np.nextafter(r, F32(0))
    return lo, hi, r


def error_bound(q, rmax, zw) -> np.ndarray:
    """The bound on |fp32 d - d| of the derivation next to screen_d, for pairs inside the domain."""
    q = np.asarray(q, np.float64)
    return 22.0 * U * q + 8.0 * U * float(rmax) * np.sqrt(q) * (1.0 + math.sqrt(zw))


def _fma(a, b, c):
    """fp32 fma(a, b, c): the product of two fp32 values is exact in float64, the sum is rounded once there first
    (a double rounding that can only matter at an exact fp32 tie)."""
    return (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(F32)


def screen_d(af, bf, rw, zw, fma=False) -> np.ndarray:
    """screen_d on fp32 (n, 3) arrays: each operation rounded (fma=False) or with the contractions fused."""
    rwf, zwf = F32(rw), F32(zw)
    with np.errstate(invalid="ignore", over="ignore"):
        t = F32(0.5) * (af[:, 1] + bf[:, 1])
        dx, dy, dz = af[:, 0] - bf[:, 0], af[:, 1] - bf[:, 1], af[:, 2] - bf[:, 2]
        if not fma:
            w = F32(1) - t * rwf
            q = dx * dx + dy * dy + zwf * (dz * dz)
        else:
            w = _fma(-t, np.full_like(t, rwf), np.ones_like(t))
            q = _fma(np.full_like(dz, zwf), dz * dz, _fma(dy, dy, dx * dx))
        return w * q


def screen_coords(w, rmax, band_only=False) -> np.ndarray:
    """The fp32 coordinates the kernels keep: screen_domain_mark puts NaN in x outside the domain."""
    w = np.asarray(w, np.float64).reshape(-1, 3)
    f = w.astype(F32)
    if not band_only:
        out = ~((np.abs(w[:, 1]) <= float(rmax)) & (np.abs(w[:, 2]) <= float(rmax)))
        f[out, 0] = np.nan
    return f


def screened(a, b, eps, rw, zw, fma=False, band_only=False) -> np.ndarray:
    """Per pair: 1 = neighbours by the fp32 screen, 0 = not neighbours by the screen, -1 = decided in float64."""
    lo, hi, rmax = screen_config(eps, rw, zw)
    d = screen_d(screen_coords(a, rmax, band_only), screen_coords(b, rmax, band_only), rw, zw, fma)
    return np.where(d > hi, 0, np.where(d < lo, 1, -1))


def decisions(a, b, eps, rw, zw, fma=False, band_only=False) -> np.ndarray:
    """The neighbour decision the kernels reach for each pair (bool)."""
    s = screened(a, b, eps, rw, zw, fma, band_only)
    ex = exact_d(a, b, rw, zw) <= eps
    return np.where(s < 0, ex, s == 1)


# ---- adversarial pairs ----------------------------------------------------------------------------------------------
@dataclass
class Cfg:
    name: str
    eps: float = 0.3
    rw: float = 0.03
    zw: float = 0.4


@dataclass
class Mount:
    name: str
    s_height: float = 1.8
    s_tilt_deg: float = -5.0
    z_max: float = 2.5


CONFIGS = [Cfg("default"), Cfg("rw0", rw=0.0), Cfg("zw0", zw=0.0), Cfg("eps_small", eps=0.05), Cfg("eps_large", eps=2.0)]
MOUNTS = [Mount("default"), Mount("high_level", s_height=2.4, s_tilt_deg=0.0, z_max=3.0)]
REPS = [None, 8, 9, 10]          # fp32 rows, int16 rows in Q8 / Q9 / Q10


def to_raw(wpt, m: Mount) -> np.ndarray:
    """World (x, y', z') -> raw sensor (x, y, z), float64 (inverse of ``world``)."""
    ang = np.radians(m.s_tilt_deg)
    c, s = np.cos(ang), np.sin(ang)
    x, yw, zw = wpt
    zr = zw - m.s_height
    return np.array([x, c * yw + s * zr, -s * yw + c * zr])


def quantize(raw, rep) -> Optional[np.ndarray]:
    """Nearest representable raw row: fp32, or the int16 lattice k / 2^Q (None if out of range)."""
    raw = np.asarray(raw, np.float64)
    if rep is None:
        return raw.astype(F32).astype(np.float64)
    k = np.rint(raw * 2.0 ** rep)
    if np.any(np.abs(k) > 32767):
        return None
    return k / 2.0 ** rep


def step_of(v, rep) -> float:
    """The spacing of representable values at v."""
    return float(np.spacing(F32(abs(v)))) if rep is None else 2.0 ** -rep


@dataclass
class Pair:
    family: str
    cfg: Cfg
    mount: Mount
    rep: Optional[int]
    a: np.ndarray            # raw rows (float64 values of the representation)
    b: np.ndarray
    target: str

    def worlds(self):
        m = self.mount
        return world(self.a, m.s_height, m.s_tilt_deg)[0], world(self.b, m.s_height, m.s_tilt_deg)[0]

    def d(self) -> float:
        wa, wb = self.worlds()
        return float(exact_d(wa, wb, self.cfg.rw, self.cfg.zw)[0])

    def neighbours(self) -> bool:
        return self.d() <= self.cfg.eps

    def rows(self, n_a: int) -> np.ndarray:
        """n_a copies of A then B as (n_a + 1, 5) rows in the representation (int16 lattice counts or float32)."""
        pts = np.concatenate([np.repeat(self.a[None], n_a, 0), self.b[None]], 0)
        if self.rep is None:
            out = np.zeros((n_a + 1, 5), np.float32)
            out[:, :3] = pts
        else:
            out = np.zeros((n_a + 1, 5), np.int16)
            out[:, :3] = np.rint(pts * 2.0 ** self.rep).astype(np.int16)
        out[:, 4] = 100
        return out


def _dist_along(cfg, m, a_raw, b_world0, direction, t, rep):
    braw = quantize(to_raw(b_world0 + t * direction, m), rep)
    if braw is None:
        return None, np.nan
    wa = world(a_raw, m.s_height, m.s_tilt_deg)
    wb = world(braw, m.s_height, m.s_tilt_deg)
    return braw, float(exact_d(wa, wb, cfg.rw, cfg.zw)[0])


def construct(cfg: Cfg, m: Mount, a_world, direction, t_range, target_d, rep, crossing=0) -> List[np.ndarray]:
    """B rows at the representable values just below and just above the ``crossing``-th (from the far end of t_range
    when negative) crossing of d(A, A + t direction) = target_d, with A = the representable row nearest a_world.
    Returns [a_raw, b_below, b_above] or [] when the crossing cannot be represented or leaves the scene."""
    a_raw = quantize(to_raw(np.asarray(a_world, np.float64), m), rep)
    if a_raw is None:
        return []
    wa = world(a_raw, m.s_height, m.s_tilt_deg)[0]
    direction = np.asarray(direction, np.float64)
    ts = np.linspace(t_range[0], t_range[1], 401)
    ds = np.array([float(exact_d(wa, wa + t * direction, cfg.rw, cfg.zw)[0]) for t in ts]) - target_d
    sign = np.nonzero(np.sign(ds[:-1]) * np.sign(ds[1:]) < 0)[0]
    if len(sign) == 0:
        return []
    k = sign[crossing]
    lo_t, hi_t = ts[k], ts[k + 1]
    f = lambda t: float(exact_d(wa, wa + t * direction, cfg.rw, cfg.zw)[0]) - target_d   # noqa: E731
    flo = f(lo_t)
    for _ in range(80):
        mid = 0.5 * (lo_t + hi_t)
        if (f(mid) > 0) == (flo > 0):
            lo_t = mid
        else:
            hi_t = mid
    b0 = quantize(to_raw(wa + lo_t * direction, m), rep)
    if b0 is None:
        return []
    # walk the representable values of the raw coordinate that moves most along `direction`
    draw = to_raw(wa + direction, m) - to_raw(wa, m)
    ax = int(np.argmax(np.abs(draw)))
    h = step_of(b0[ax], rep)

    def dd(k):
        b = b0.copy()
        b[ax] += k * h
        if rep is None:
            b[ax] = float(F32(b[ax]))
        wb = world(b, m.s_height, m.s_tilt_deg)
        return b, float(exact_d(wa[None], wb, cfg.rw, cfg.zw)[0])

    k = 0
    b, d = dd(0)
    up = (dd(1)[1] > d) == (draw[ax] > 0)          # does a step along +ax move d the way +direction does
    sgn = 1 if up else -1
    # step until d(k) <= target < d(k + sgn) (the rows straddle target_d in the representation)
    for _ in range(100000):
        b1, d1 = dd(k + sgn)
        if d <= target_d < d1 or d1 <= target_d < d:
            break
        k += sgn if (d <= target_d) == (d < d1) else -sgn
        b, d = dd(k)
    else:
        return []
    lo_b, hi_b = (b, b1) if d <= target_d else (b1, b)
    out = []
    for bb in (lo_b, hi_b):
        if rep is not None and np.any(np.abs(np.rint(bb * 2.0 ** rep)) > 32767):
            return []
        if not in_scene(world(bb, m.s_height, m.s_tilt_deg), m.z_max)[0]:
            return []
        out.append(bb)
    if not in_scene(world(a_raw, m.s_height, m.s_tilt_deg), m.z_max)[0]:
        return []
    return [a_raw] + out


def _families(cfg: Cfg, m: Mount):
    """(name, A world, direction, t range, crossing) of each family for a configuration and mounting."""
    zmid = min(0.9, 0.5 * m.z_max)
    out = [("near_x", (0.3, 2.0, zmid), (1, 0, 0), (0.0, 4.0), 0),
           ("near_y", (0.3, 2.0, zmid), (0, 1, 0), (0.0, 4.0), 0),
           ("y20_x", (-0.4, 20.0, zmid), (1, 0, 0), (0.0, 8.0), 0),
           ("y20_y", (-0.4, 20.0, zmid), (0, 1, 0), (0.0, 8.0), 0)]
    if cfg.rw > 0:
        y0 = 1.0 / cfg.rw                              # w = 0 at mean y' = y0
        out += [("w0_dx", (-54.0, y0 - 0.05, zmid), (1, 0, 0), (0.0, 120.0), 0),
                ("w0_dy", (0.2, y0 - 13.0, zmid), (0, 1, 0), (0.0, 27.0), -1)]
    else:
        out += [("far_dy", (0.2, 6000.0, zmid), (0, 1, 0), (0.0, 4.0), 0)]
    return out


def adversarial_pairs(configs=CONFIGS, mounts=MOUNTS, reps=REPS) -> List[Pair]:
    """For each configuration, mounting, representation and family: the pairs straddling d = eps, eps -/+ band / 2
    (inside the band) and eps -/+ 1.5 band (just outside it)."""
    pairs = []
    for cfg in configs:
        band = 1e-3 * cfg.eps + 1e-4
        for m in mounts:
            for rep in reps:
                for name, aw, direc, tr, cross in _families(cfg, m):
                    for tname, target in (("eps", cfg.eps), ("in_lo", cfg.eps - 0.5 * band),
                                          ("in_hi", cfg.eps + 0.5 * band), ("out_lo", cfg.eps - 1.5 * band),
                                          ("out_hi", cfg.eps + 1.5 * band)):
                        got = construct(cfg, m, aw, direc, tr, target, rep, cross)
                        for k, side in ((1, "below"), (2, "above")):
                            if got:
                                pairs.append(Pair(name, cfg, m, rep, got[0], got[k], "%s_%s" % (tname, side)))
                p = wneg_pair(cfg, m, rep) if cfg.rw > 0 else None
                if p is not None:
                    pairs.append(p)
    return pairs


def wneg_pair(cfg: Cfg, m: Mount, rep) -> Optional[Pair]:
    """A pair 100 m apart in x whose mean y' puts the float64 w just below 0: d <= 0, so neighbours, while fp32 w can
    come out positive and d_f far above eps."""
    y0 = 1.0 / cfg.rw
    zmid = min(0.9, 0.5 * m.z_max)
    a = quantize(to_raw((-50.0, y0, zmid), m), rep)
    if a is None:
        return None
    wa = world(a, m.s_height, m.s_tilt_deg)[0]
    b0 = quantize(to_raw((50.0, wa[1], wa[2]), m), rep)
    if b0 is None:
        return None
    h = step_of(b0[1], rep)
    for k in range(-200, 200):
        b = b0.copy()
        b[1] += k * h
        wb = world(b, m.s_height, m.s_tilt_deg)[0]
        w64 = 1.0 - ((wa[1] + wb[1]) * 0.5) * cfg.rw
        if w64 < 0 and in_scene(wb, m.z_max)[0] and in_scene(wa, m.z_max)[0]:
            return Pair("wneg", cfg, m, rep, a, b, "w_below_0")
    return None


def random_domain(n, rng, cfg: Cfg, m: Mount, rep=None):
    """Seeded pairs of the admitted domain: x, y' up to the Q8 range (128 m), 0 < z' <= z_max, mostly close pairs
    (so that many fall near eps) scattered over the whole range of y'."""
    ax = rng.uniform(-120, 120, n)
    ay = rng.uniform(0, 127, n)
    az = rng.uniform(1e-3, m.z_max, n)
    r = np.sqrt(cfg.eps / 0.05) * rng.uniform(0, 1, n) ** 2
    th = rng.uniform(0, 2 * np.pi, n)
    ph = rng.uniform(-1, 1, n)
    bx, by, bz = ax + r * np.cos(th), ay + r * np.sin(th), np.clip(az + 0.3 * ph, 1e-3, m.z_max)
    A = np.stack([to_raw(p, m) for p in zip(ax, ay, az)])
    B = np.stack([to_raw(p, m) for p in zip(bx, by, bz)])
    lim = 127.9 if rep is None else 32767 / 2.0 ** rep       # int16 rows: what the lattice can hold
    A, B = quantize(np.clip(A, -lim, lim), rep), quantize(np.clip(B, -lim, lim), rep)
    wa, wb = world(A, m.s_height, m.s_tilt_deg), world(B, m.s_height, m.s_tilt_deg)
    ok = in_scene(wa, m.z_max) & in_scene(wb, m.z_max)
    return wa[ok], wb[ok]


def w0_search(cfg: Cfg, m: Mount, rep, n, rng) -> List[Pair]:
    """The w -> 0 family made adversarial: pairs about 100 m apart in x (or with a large dy when ``dy``) whose mean y'
    puts w near 0, B's x placed at the representable values around d = eps.  Returns the pairs on which the band-only
    rule decides wrongly under either contraction (the pairs that need the domain)."""
    y0 = 1.0 / cfg.rw
    zmax = m.z_max
    ya = y0 + rng.uniform(-0.4, 0.4, n)
    yb = 2 * y0 - ya + rng.uniform(-0.3, 0.1, n)
    za, zb = rng.uniform(0.1, zmax - 0.1, n), rng.uniform(0.1, zmax - 0.1, n)
    A = np.stack([to_raw((-50.0, a, c), m) for a, c in zip(ya, za)])
    B = np.stack([to_raw((0.0, b, c), m) for b, c in zip(yb, zb)])
    A, B = quantize(A, rep), quantize(B, rep)
    if A is None or B is None:
        return []
    wa, wb = world(A, m.s_height, m.s_tilt_deg), world(B, m.s_height, m.s_tilt_deg)
    w = 1.0 - ((wa[:, 1] + wb[:, 1]) * 0.5) * cfg.rw
    rest = (wa[:, 1] - wb[:, 1]) ** 2 + cfg.zw * (wa[:, 2] - wb[:, 2]) ** 2
    with np.errstate(invalid="ignore", divide="ignore"):
        dx = np.sqrt(cfg.eps / w - rest)
    ok = (w > 0) & np.isfinite(dx) & (dx < 120)
    out = []
    for i in np.nonzero(ok)[0]:
        for k in range(-2, 3):
            b = B[i].copy()
            b[0] = A[i, 0] + dx[i]
            q = quantize(b, rep)
            if q is None:
                continue
            b[0] = q[0] + k * step_of(q[0], rep)
            if rep is not None and abs(b[0]) * 2.0 ** rep > 32767:
                continue
            wbb = world(b, m.s_height, m.s_tilt_deg)
            if not (in_scene(wa[i], zmax)[0] and in_scene(wbb, zmax)[0]):
                continue
            ex = exact_d(wa[i], wbb, cfg.rw, cfg.zw)[0] <= cfg.eps
            if any(decisions(wa[i], wbb, cfg.eps, cfg.rw, cfg.zw, f, True)[0] != ex for f in (False, True)):
                out.append(Pair("w0_search", cfg, m, rep, A[i], b, "band_only_wrong"))
    return out

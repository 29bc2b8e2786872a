"""The pose network's kernels layer by layer against a float64 reference of their split-bf16 arithmetic
(tests/pose_reference.py), at the row counts and tile edges where the kernels change behaviour.

Each run reads the network's intermediates back with the mmw_pose_intermediate test hook and checks every layer from the
previous layer's kernel output: |kernel - emulation| <= TAU M, |kernel - exact float64| <= TAU_EXACT M, every (hi, lo)
pair a valid round-to-nearest split, and the input layer the exact split of the fp32 feature maps.  A failure names the
layer, the row and the (d, h, w, c) of the worst element.

TAU is about four times the worst ratio measured on an NVIDIA B200 over every test of this file (DESIGN.md section 2);
the mistakes a kernel rewrite plausibly makes sit far above it (test_checker_rejects_emulated_mutants).  Set
MMW_POSE_RATIO_LOG=<file.json> to record the worst ratios of a run, per check and layer, when the kernels change.
"""
import ctypes
import json
import os
import re

import numpy as np
import pytest
import torch

import pose_reference as pr
from helpers import KEYPOINT_ATOL
from mmwave_msc_b200 import _lib, pose_weights as pw, synth
from mmwave_msc_b200.batched import BatchedTracker, default_config
from oracle import mmw_oracle as mo

# Bounds per layer (1 conv 1, 2 conv 2 + BN 1, 3 dense 1 + BN 2, 4 dense 2) in units of M, about four times the worst
# ratio measured on an NVIDIA B200 (1000 W power limit) over every test of this file; DESIGN.md section 2 has the figures.
TAU = {1: 2.0 ** -17.5, 2: 2.0 ** -17, 3: 2.0 ** -14.5, 4: 2.0 ** -18}             # against the emulation
TAU_EXACT = {1: 2.0 ** -13.75, 2: 2.0 ** -14.25, 3: 2.0 ** -14.5, 4: 2.0 ** -15.5}  # against exact float64
# the root mean square over a layer is a stable statistic: about 2.4 times the worst measured, so that one dense-1 K block
# without its a_lo w_hi product (2^-18.0 in test_checker_rejects_emulated_mutants) stays outside
TAU_RMS = {1: 2.0 ** -24.25, 2: 2.0 ** -23.75, 3: 2.0 ** -18.5, 4: 2.0 ** -20.75}
TAU_E2E = 2.0 ** -20        # keypoints against pose_forward, in units of the magnitude carried through all layers
TAU_FP32 = 2.0 ** -19       # CUDA-core fp32 path against exact float64

_RATIOS = {}


def _record(kind, variant, stats):
    for l, vals in stats.items():
        key = "%s/%s/layer %d" % (kind, "3d" if variant == pw.VARIANT_3D else "2d", l)
        old = _RATIOS.get(key, [0.0] * len(vals))
        _RATIOS[key] = [max(a, float(b)) for a, b in zip(old, vals)]


@pytest.fixture(scope="module", autouse=True)
def _ratio_log():
    yield
    path = os.environ.get("MMW_POSE_RATIO_LOG")
    if path:
        with open(path, "w") as f:
            json.dump({k: [float(np.log2(x)) if x > 0 else None for x in v] for k, v in sorted(_RATIOS.items())}, f,
                      indent=1)


@pytest.fixture(autouse=True)
def _plain_kernels(monkeypatch):
    # MMW_GEMM_DBG / MMW_FEAT_DBG leave work out (timing experiments); MMW_FC1_BN forces a dense-1 tile width
    for k in ("MMW_GEMM_DBG", "MMW_FEAT_DBG", "MMW_FC1_BN"):
        monkeypatch.delenv(k, raising=False)


def _dev():
    return "cuda" if torch.cuda.is_available() else "cpu"


def _fb(variant):
    return 2 if variant == pw.VARIANT_3D else 0


def _tracker(variant, n_cap, W):
    bt = BatchedTracker((n_cap + 7) // 8, max_tracks=8, config=default_config(frames_batch=_fb(variant)))
    bt.load_pose_weights(W, variant)
    return bt


def make_feats(rng, n, variant, wide=False):
    """Feature maps like format_single_frame's: 20-64 points per frame sorted by x, zero pad rows after them.  wide:
    also frames without points, peakVal up to 65 535 and rows whose values are exact in bf16 (lo = 0)."""
    nfr = _fb(variant) + 1
    feats = np.zeros((n, nfr, 64, 5), np.float32)
    for i in range(n):
        for f in range(nfr):
            k = int(rng.integers(0 if wide else 20, 65))
            rows = np.zeros((64, 5), np.float32)
            rows[:k, 0] = rng.normal(0, 0.15, k); rows[:k, 1] = rng.normal(0, 0.15, k)
            rows[:k, 2] = rng.normal(1.0, 0.4, k); rows[:k, 3] = rng.normal(0, 0.3, k)
            peak = np.floor(rng.gamma(0.5, 54.0, k)) + 1
            if wide:
                big = rng.random(k) < 0.2
                peak[big] = rng.integers(1000, 65536, int(big.sum()))
            rows[:k, 4] = (peak - 27.0187) / 70.351
            if wide and rng.random() < 0.25:
                rows = pr.bf16_value(pr.bf16_rn(rows)).numpy().astype(np.float32)
            feats[i, f] = rows[np.argsort(rows[:, 0], kind="stable")]
    return feats.reshape((n, nfr, 8, 8, 5) if nfr == 3 else (n, 8, 8, 5))


def wide_weights(variant, seed=9):
    """make_pose_weights with per-channel power-of-two scales on every kernel and BatchNorm variances near 0 (|scale|
    up to about 30) on a quarter of the channels."""
    rng = np.random.default_rng(seed)
    W = [w.copy() for w in pw.make_pose_weights(variant, seed)]
    for i in (0, 2, 8, 14):
        W[i] *= (2.0 ** rng.integers(-3, 4, size=W[i].shape[-1])).astype(np.float32)
    for i in (7, 13):
        k = len(W[i]) // 4
        W[i][:k] = rng.uniform(0, 1e-5, k)
    return [np.ascontiguousarray(w, np.float32) for w in W]


WEIGHTS = {"seed7": lambda v: pw.make_pose_weights(v, 7), "seed8": lambda v: pw.make_pose_weights(v, 8),
           "wide": wide_weights}


def run_layers(bt, feats):
    """mmw_pose on feats, then the kernel outputs check_layers takes."""
    kp = bt.pose(feats)
    outs = {l: bt.pose_intermediate(l) for l in range(4)}
    outs[4] = kp
    assert all(len(outs[l][0]) == len(feats) for l in range(4))
    return outs


def check(net, feats, outs, kind, variant, tag, layers=(0, 1, 2, 3, 4)):
    st = pr.check_layers(net, feats, outs, TAU, TAU_EXACT, TAU_RMS, tag=tag, layers=layers)
    _record(kind, variant, st)
    return st


def check_e2e(net, W, feats, kp, variant, kind, absolute=True):
    """Keypoints against the exact float64 forward pass: within TAU_E2E of the magnitude carried through the layers,
    and (trained-like weights) within today's 1 mm."""
    ref, mag = net.exact_chain(feats)[4]
    got = net.t64(kp)
    r = pr.check_bound(4, got, ref, mag, TAU_E2E, "exact float64", "end to end: ")
    _record(kind + "/e2e", variant, {4: (r,)})
    if absolute:
        err = np.abs(kp - mo.pose_forward(W, feats, np.float64)).max()
        assert err < KEYPOINT_ATOL, "max joint error %.3g m" % err
    assert float(ref.abs().mean()) > 0.05          # not vacuous


# ---- (a) per-layer parity, both variants, three weight sets ----------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("wset", ["seed7", "seed8", "wide"])
@pytest.mark.parametrize("variant", [pw.VARIANT_3D, pw.VARIANT_2D])
def test_layers_match_split_bf16_reference(variant, wset):
    W = WEIGHTS[wset](variant)
    net = pr.PoseNet(W, _dev())
    feats = make_feats(np.random.default_rng(21), 200, variant, wide=wset == "wide")
    bt = _tracker(variant, 512, W)
    outs = run_layers(bt, feats)
    check(net, feats, outs, "parity", variant, "%s: " % wset)
    check_e2e(net, W, feats, outs[4], variant, "parity", absolute=wset != "wide")


# ---- (b) row-count edges -----------------------------------------------------------------------------------------
# 3-D: dense 2's 128-row tiles, dense 1's 256-row CTA pairs (257: a pair whose second CTA has no rows), and 148 * 8 + 1
# samples so that every conv CTA goes round its slab ring (8 / 4 slots) and its two TMEM buffers several times.
# 2-D: three samples per slab, remainders 0, 1, 2 of n mod 3, and >= 8 slabs per conv CTA with n mod 3 = 1 and 2.
EDGES = {pw.VARIANT_3D: [148 * 8 + 1, 385, 257, 256, 255, 129, 128, 127, 2, 1],
         pw.VARIANT_2D: [148 * 24 + 2, 148 * 24 + 1, 5, 4, 3, 2, 1]}


@pytest.mark.gpu
@pytest.mark.parametrize("variant", [pw.VARIANT_3D, pw.VARIANT_2D])
def test_row_count_edges(variant):
    """Largest n first, so every smaller run also sees the stale rows of a larger one; every run's rows must equal the
    same rows of the largest run bit for bit (a row's result does not depend on the batch around it)."""
    W = pw.make_pose_weights(variant, 7)
    net = pr.PoseNet(W, _dev())
    ns = EDGES[variant]
    cap = (max(ns) + 7) // 8 * 8
    feats = make_feats(np.random.default_rng(22), max(ns), variant)
    bt = _tracker(variant, cap, W)
    first = None
    for n in ns:
        outs = run_layers(bt, feats[:n])
        check(net, feats[:n], outs, "edges", variant, "n = %d: " % n)
        if first is None:
            first = outs
            continue
        for l in range(4):
            for p in range(2):
                assert np.array_equal(outs[l][p], first[l][p][:n]), "n = %d: %s differs from the same rows at n = %d" % (
                    n, pr.LAYER_NAMES[l], ns[0])
        assert np.array_equal(outs[4], first[4][:n]), "n = %d: keypoints differ" % n
    with pytest.raises(_lib.MmwError, match="error -3"):          # MMW_ERR_CAPACITY
        bt.pose(np.zeros((cap + 1,) + feats.shape[1:], np.float32))


# ---- (c) dense 1 tile widths -------------------------------------------------------------------------------------
FC1_ROWS = [3073, 3072, 2305, 2304, 2049, 2048, 2047, 257, 256, 255]


@pytest.mark.gpu
def test_dense1_tile_widths_against_reference(monkeypatch):
    """MMW_FC1_BN forces 256 x 176 (the last of the 9 column tiles is 128 wide, its W rows the tensor map's out-of-bounds
    zeros), 256 x 192 and 256 x 256 tiles.  Dense 1 passes the bound at every width and row count, and the three widths
    give the same bits."""
    variant = pw.VARIANT_3D
    W = pw.make_pose_weights(variant, 7)
    net = pr.PoseNet(W, _dev())
    feats = make_feats(np.random.default_rng(23), max(FC1_ROWS), variant)
    base = None
    for bn in ("176", "192", "256"):
        monkeypatch.setenv("MMW_FC1_BN", bn)          # read when the weights are loaded
        bt = _tracker(variant, 4096, W)
        for n in FC1_ROWS:
            outs = run_layers(bt, feats[:n])
            check(net, feats[:n], outs, "fc1 tiles", variant, "BN %s, n = %d: " % (bn, n), layers=(3,))
            if base is None:
                base = outs
            for l in (2, 3):
                for p in range(2):
                    assert np.array_equal(outs[l][p], base[l][p][:n]), "BN %s, n = %d: %s" % (bn, n, pr.LAYER_NAMES[l])
            assert np.array_equal(outs[4], base[4][:n]), "BN %s, n = %d: keypoints" % (bn, n)
        bt.close()


# ---- (d) dense 2 around its K-split switch -----------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n", [16384, 16385])
def test_dense2_k_split_switch(n):
    """16 384 rows: dense 2 as 4-CTA clusters splitting K; 16 385: the unsplit kernel.  The rows are copies of 300
    distinct feature maps at varied positions: the reference runs on the distinct rows, and every copy of a row must
    equal every other copy bit for bit, in every layer."""
    variant = pw.VARIANT_3D
    W = pw.make_pose_weights(variant, 7)
    net = pr.PoseNet(W, _dev())
    rng = np.random.default_rng(24)
    distinct = make_feats(rng, 300, variant)
    which = np.concatenate([np.arange(300), rng.integers(0, 300, n - 300)])
    rng.shuffle(which)
    bt = _tracker(variant, 16640, W)
    outs = run_layers(bt, distinct[which])
    first = np.full(300, -1)
    for i in range(n - 1, -1, -1):
        first[which[i]] = i
    rep = first[which]                                  # the first copy of each row's feature map
    for l in range(4):
        for p in range(2):
            same = (outs[l][p] == outs[l][p][rep]).all(axis=1)
            assert same.all(), "%s: row %d differs from its copy at row %d" % (
                pr.LAYER_NAMES[l], int(np.argmin(same)), rep[int(np.argmin(same))])
    same = (outs[4] == outs[4][rep]).all(axis=1)
    assert same.all(), "keypoints: row %d differs from its copy at row %d" % (int(np.argmin(same)), rep[np.argmin(same)])
    sub = {l: (outs[l][0][first], outs[l][1][first]) for l in range(4)}
    sub[4] = outs[4][first]
    check(net, distinct, sub, "dense2 split", variant, "n = %d: " % n)


# ---- (e) stale rows ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_no_leakage_from_stale_rows():
    """n = 3000 then n = 5 in one context: the 5 rows equal those of a fresh context, bit for bit, in every layer; and
    the other way round."""
    variant = pw.VARIANT_3D
    W = pw.make_pose_weights(variant, 7)
    rng = np.random.default_rng(25)
    big, small = make_feats(rng, 3000, variant), make_feats(rng, 5, variant)
    a, b = _tracker(variant, 4096, W), _tracker(variant, 4096, W)
    a_big, a_small = run_layers(a, big), run_layers(a, small)
    b_small, b_big = run_layers(b, small), run_layers(b, big)
    for got, want, what in ((a_small, b_small, "5 rows after 3000"), (b_big, a_big, "3000 rows after 5")):
        for l in range(4):
            for p in range(2):
                assert np.array_equal(got[l][p], want[l][p]), "%s: %s" % (what, pr.LAYER_NAMES[l])
        assert np.array_equal(got[4], want[4]), what + ": keypoints"


# ---- (f) the step path against the stage path ---------------------------------------------------------------------------
def _row_order(feats_sorted, in_hi, in_lo):
    """Index into the (scene, track)-sorted rows of every row of the run, found by its packed input; raises when a row
    of the run is not the exact split of any returned feature map."""
    n = len(feats_sorted)
    hi, lo = (x.numpy().view(np.uint16) for x in pr.split(feats_sorted.reshape(n, -1)))
    keys = {}
    for i in range(n):
        keys.setdefault(hi[i].tobytes() + lo[i].tobytes(), []).append(i)
    perm = np.zeros(n, np.int64)
    for j in range(n):
        cand = keys.get(in_hi[j].tobytes() + in_lo[j].tobytes())
        assert cand, "%s: row %d of the step's network input is not the split of any pose row" % (pr.LAYER_NAMES[0], j)
        perm[j] = cand.pop()
    return perm


@pytest.mark.gpu
@pytest.mark.parametrize("variant", [pw.VARIANT_3D, pw.VARIANT_2D])
def test_step_path_equals_stage_path(variant):
    """Serial mmw_step with MMW_STEP_POSE: pose_feature_kernel writes the network input itself (not pack_input_kernel).
    It must be the exact split of the rows mmw_get_pose_rows returns, every layer must pass the bound, and every live
    track's keypoints must equal what mmw_pose gives for the same rows, bit for bit (S * max_tracks <= 16 384, so both
    paths run the same dense 2 kernel)."""
    S, F = 48, 24
    W = pw.make_pose_weights(variant, 7)
    net = pr.PoseNet(W, _dev())
    cfg = default_config(frames_batch=_fb(variant))
    bt, stage = BatchedTracker(S, config=cfg), BatchedTracker(S, config=cfg)
    bt.load_pose_weights(W, variant); stage.load_pose_weights(W, variant)
    checked = 0
    for f, b in enumerate(synth.gen_batch(list(range(300, 300 + S)), F)):
        bt.step(b.points, b.offsets, b.dt, pose=True)
        if f < 8 or f % 4:
            continue
        outs = {l: bt.pose_intermediate(l) for l in range(4)}
        si, ti, feats = bt.pose_rows()
        n = len(si)
        assert len(outs[0][0]) == n and n > S
        perm = _row_order(feats, *outs[0])
        tr, _ = bt.tracks()
        kp_step = tr["keypoints"][si[perm], ti[perm]]
        kp_stage = stage.pose(feats[perm])
        assert kp_step.tobytes() == kp_stage.tobytes(), "frame %d: step keypoints differ from mmw_pose" % f
        outs[4] = kp_step
        check(net, feats[perm], outs, "step", variant, "frame %d: " % f)
        checked += 1
    assert checked >= 4


# ---- (g) the CUDA-core path --------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("variant", [pw.VARIANT_3D, pw.VARIANT_2D])
def test_cuda_core_path_layers(variant):
    """set_dense_path(False): conv 2 (+ BN 1) against the exact float64 chain from the feature maps, dense 1 (+ BN 2) and
    dense 2 against exact float64 from the kernel's own previous layer, in units of M with an fp32 bound."""
    W = pw.make_pose_weights(variant, 7)
    net = pr.PoseNet(W, _dev())
    feats = make_feats(np.random.default_rng(26), 200, variant)
    bt = _tracker(variant, 512, W)
    bt.set_dense_path(False)
    kp = bt.pose(feats)
    l2, l3 = bt.pose_intermediate(2, tensor_cores=False), bt.pose_intermediate(3, tensor_cores=False)
    with pytest.raises(_lib.MmwError, match="error -1"):
        bt.pose_intermediate(1, tensor_cores=False)
    ref2, mag2 = (x.reshape(len(feats), -1) for x in net.exact_chain(feats)[2])
    st = {2: pr.check_bound(2, net.t64(l2), ref2, mag2, TAU_FP32, "exact float64", "CUDA-core path: ")}
    for l, got, prev in ((3, l3, l2), (4, kp, l3)):
        a = net.t64(prev)
        _, exact, mag = net.layer(l, a, torch.zeros_like(a))
        st[l] = pr.check_bound(l, net.t64(got), exact, mag, TAU_FP32, "exact float64", "CUDA-core path: ")
    _record("cuda cores", variant, {l: (r,) for l, r in st.items()})


# ---- the hook's refusals -------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_intermediate_hook_refusals():
    """MMW_ERR_STATE without weights, before any run, and after a throughput-mode step (its intermediates belong to a
    frame that may still be in flight); the next serial step makes them readable again."""
    W = pw.make_pose_weights(pw.VARIANT_3D, 7)
    bt = BatchedTracker(16)
    with pytest.raises(_lib.MmwError, match="error -4"):
        bt.pose_intermediate(0)
    bt.load_pose_weights(W)
    with pytest.raises(_lib.MmwError, match="error -4"):
        bt.pose_intermediate(0)
    batches = synth.gen_batch(list(range(16)), 6)
    for b in batches[:5]:
        bt.step(b.points, b.offsets, b.dt, pose=True, pipeline=True)
    bt.sync()
    with pytest.raises(_lib.MmwError, match="error -4"):
        bt.pose_intermediate(3)
    b = batches[5]
    bt.step(b.points, b.offsets, b.dt, pose=True)
    hi, lo = bt.pose_intermediate(3)
    assert len(hi) == len(bt.pose_rows()[0]) > 0
    n = ctypes.c_int(0)
    assert bt.lib.mmw_pose_intermediate(bt._h, 4, ctypes.byref(n), None, 0) == -1          # no layer 4
    assert bt.lib.mmw_pose_intermediate(bt._h, 3, ctypes.byref(n), _lib.ptr(hi), hi.nbytes) == -3   # too small


# ---- (h) the checker itself, on emulated builds (CPU) ------------------------------------------------------------------
@pytest.mark.parametrize("mutation", [None] + sorted(pr.MUTATIONS))
def test_checker_rejects_emulated_mutants(mutation):
    """A build emulated on the CPU with fp32 accumulation passes the per-layer check; each mistake a kernel rewrite can
    plausibly make, and that today's 1 mm end-to-end bar lets through, fails it at the layer that has it."""
    W = pw.make_pose_weights(pw.VARIANT_3D, 7)
    net = pr.PoseNet(W)
    feats = make_feats(np.random.default_rng(27), 64, pw.VARIANT_3D)
    outs = pr.emulated_build(net, feats, mutation)
    if mutation is None:
        st = pr.check_layers(net, feats, outs, TAU, TAU_EXACT, TAU_RMS)
        assert all(st[l][0] <= TAU[l] / 4 for l in TAU)             # the emulation is not at the edge of the bound
        return
    with pytest.raises(AssertionError, match="^" + re.escape(pr.LAYER_NAMES[pr.MUTATIONS[mutation]])):
        pr.check_layers(net, feats, outs, TAU, TAU_EXACT, TAU_RMS)

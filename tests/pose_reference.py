"""Float64 reference of the pose network as the tensor-core kernels compute it, layer by layer, and the per-layer bound.

The tensor-core kernels (mmwave_msc_b200/csrc/pose_tc.cu) split every fp32 operand into two bf16 terms, a = a_hi + a_lo,
w = w_hi + w_lo, and accumulate the three products a_hi*w_hi + a_lo*w_hi + a_hi*w_lo in fp32.  Each layer's epilogue adds
the bias, applies ReLU and (conv 2, dense 1) BatchNorm as scale*v + shift with the fp32 constants mmw_load_pose_weights
folds, and writes the next layer's operand split again.  Here each layer is evaluated from the previous layer's KERNEL
output (hi + lo decoded exactly), so a failure points at the layer that went wrong:

  emulation : the three products in float64, then bias, ReLU and the folded fp32 BatchNorm constants
  exact     : the same layer in float64 from the fp32 weights (oracle.mmw_oracle.pose_forward semantics)
  M         : sum |a| |w| + |bias| per output element; |scale| M + |shift| after BatchNorm

and a kernel output passes when |kernel - emulation| <= tau M and |kernel - exact| <= tau_exact M, beyond what the
rounding of its own split output accounts for (split_allowance), and when every (hi, lo) pair is a valid split.  Layers:
  0 network input (split of the fp32 feature maps)   1 conv 1 + ReLU   2 conv 2 + ReLU + BN 1   3 dense 1 + ReLU + BN 2
  4 dense 2 (fp32 keypoints, not split)
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn.functional as Fn

LAYER_NAMES = {0: "input split", 1: "conv 1", 2: "conv 2 + BN 1", 3: "dense 1 + BN 2", 4: "dense 2"}


# ---- bf16 split ------------------------------------------------------------------------------------------------
# Everything below works on torch tensors on any device (the GPU tests evaluate the float64 reference on the GPU, where
# the dense-1 products of a few thousand rows take milliseconds); bf16 values travel as their uint16 bits in int16.
def _t(x, device=None, dtype=None):
    if isinstance(x, torch.Tensor):
        return x.to(device=device or x.device, dtype=dtype or x.dtype)
    a = np.ascontiguousarray(x)
    if a.dtype == np.uint16:
        a = a.view(np.int16)
    return torch.from_numpy(a).to(device=device, dtype=dtype)


def bf16_rn(x):
    """Bits (int16) of the round-to-nearest-even bf16 of float32(x) (torch's float32 -> bfloat16 cast)."""
    return _t(x, dtype=torch.float32).to(torch.bfloat16).view(torch.int16)


def bf16_value(bits):
    """float64 value of bf16 bits (exact)."""
    b = _t(bits).to(torch.int32) & 0xFFFF
    return (b << 16).view(torch.float32).to(torch.float64)


def split(x):
    """(hi, lo) bits as split2 in pose_tc.cu and f2bf on the host compute them: hi = bf16(x), lo = bf16(x - hi)."""
    x32 = _t(x, dtype=torch.float32)
    hi = bf16_rn(x32)
    return hi, bf16_rn(x32 - bf16_value(hi).to(torch.float32))


def split_trunc(x):
    """A WRONG split, by truncation instead of rounding (for the checker's self-test)."""
    x32 = _t(x, dtype=torch.float32)
    hi = (x32.view(torch.int32) >> 16).to(torch.int16)
    r = x32 - bf16_value(hi).to(torch.float32)
    return hi, (r.view(torch.int32) >> 16).to(torch.int16)


def decode(hi, lo):
    return bf16_value(hi) + bf16_value(lo)


def _half_ulp(v):
    """Half a bf16 ulp of bf16 values v (0 where v is 0): |v| = m 2^e with m in [0.5, 1), an ulp is 2^(e - 8)."""
    _, e = torch.frexp(v)
    return torch.where(v == 0, torch.zeros_like(v), torch.ldexp(torch.ones_like(v), e - 9))


def split_violations(hi, lo):
    """Mask of (hi, lo) pairs no round-to-nearest split can produce: |lo| must not exceed half a bf16 ulp of hi (and lo
    must be 0 where hi is 0).  A truncating split breaks this for about half of its values.  (bf16_rn(hi + lo) == hi is
    not an invariant of a correct split: when x - hi rounds up to exactly half an ulp, hi + lo is a tie that may round
    to the even neighbour of hi.)"""
    return bf16_value(lo).abs() > _half_ulp(bf16_value(hi))


def split_allowance(hi, lo):
    """What rounding the epilogue's fp32 value and splitting it may add to a correct kernel's output, per element: half a
    bf16 ulp of lo (hi + lo misses the fp32 value by at most that) plus half an fp32 ulp of the value.  It is relative to
    the output, not to M, and would otherwise set the floor of the ratios (about 2^-17 of the output)."""
    h, l = bf16_value(hi), bf16_value(lo)
    return _half_ulp(l) + (h + l).abs() * 2.0 ** -24


# ---- the network's constants --------------------------------------------------------------------------------------
def folded_bn(gamma, beta, mean, var):
    """scale, shift as mmw_load_pose_weights folds them, in fp32: s = gamma / sqrt(var + 1e-3), t = beta - mean s."""
    g, b, m, v = (np.asarray(a, np.float32) for a in (gamma, beta, mean, var))
    s = (g / np.sqrt(v + np.float32(1e-3))).astype(np.float32)
    t = (b - m * s).astype(np.float32)
    return s, t


class PoseNet:
    """The weights of one network (Keras get_weights() order) prepared for the per-layer references on `device`."""

    def __init__(self, weights, device="cpu"):
        w = [np.asarray(a, np.float32) for a in weights]
        self.device = torch.device(device)
        self.D = 3 if w[0].ndim == 5 else 1
        k1, k2 = w[0], w[2]
        if self.D == 1:                                  # the 2-D net as a 3-D one with depth 1
            k1, k2 = k1[None], k2[None]
        self.k = [k1, k2]                                # (kd, kh, kw, cin, cout)
        self.b = [w[1], w[3], w[9], w[15]]
        self.wd = [w[8], w[14]]                          # (in, out)
        self.bn_f32 = [folded_bn(*w[4:8]), folded_bn(*w[10:14])]
        self.bn_raw = [w[4:8], w[10:14]]
        self.Kf, self.H = w[8].shape

    def t64(self, x):
        return _t(x, self.device, torch.float64)

    def _conv(self, x, k):
        """x (n, D, 8, 8, cin), k (kd, kh, kw, cin, cout): 'same' cross-correlation -> (n, D, 8, 8, cout)."""
        pad = (1, 1, 1) if self.D == 3 else (0, 1, 1)
        return Fn.conv3d(x.permute(0, 4, 1, 2, 3), k.permute(4, 3, 0, 1, 2), padding=pad).permute(0, 2, 3, 4, 1)

    @staticmethod
    def _mm(a, w):
        return a @ w

    def layer(self, l, a_hi, a_lo):
        """(emulation, exact, M) of layer l = 1..4 from the previous layer's kernel output, given as float64 tensors of
        the values of hi and lo (conv layers: (n, D, 8, 8, cin); dense layers: (n, K))."""
        a = a_hi + a_lo
        conv = l <= 2
        w = self.k[l - 1] if conv else self.wd[l - 3]
        op = self._conv if conv else self._mm
        wh, wl = (bf16_value(b).to(self.device) for b in split(w))
        w64 = self.t64(w)
        with torch.no_grad():
            # a_hi w_hi + a_lo w_hi = a w_hi: the products of bf16 values are exact in float64
            pre_emu = op(a, wh) + op(a_hi, wl)
            pre_exact = op(a, w64)
            mag = op(a.abs(), w64.abs())
        bias = self.t64(self.b[l - 1])
        mag = mag + bias.abs()
        if l == 4:
            return pre_emu + bias, pre_exact + bias, mag
        v_emu, v_exact = torch.relu(pre_emu + bias), torch.relu(pre_exact + bias)
        if l == 1:
            return v_emu, v_exact, mag
        s, t = (self.t64(c) for c in self.bn_f32[l - 2])
        g, be, mu, var = (self.t64(c) for c in self.bn_raw[l - 2])
        return v_emu * s + t, (v_exact - mu) / torch.sqrt(var + 1e-3) * g + be, s.abs() * mag + t.abs()

    def exact_chain(self, feats):
        """Exact float64 forward pass from fp32 feature maps, with the magnitudes carried through the layers (the
        error bound of a path whose intermediate layers cannot be read back): {layer: (value, M)} for layers 1..4."""
        x = self.t64(np.asarray(feats, np.float32)).reshape(-1, self.D, 8, 8, 5)
        out, m = {}, x.abs()
        with torch.no_grad():
            for l in (1, 2, 3, 4):
                if l == 3:
                    x, m = x.reshape(len(x), -1), m.reshape(len(m), -1)
                w = self.t64(self.k[l - 1] if l <= 2 else self.wd[l - 3])
                op = self._conv if l <= 2 else self._mm
                b = self.t64(self.b[l - 1])
                x, m = op(x, w) + b, op(m, w.abs()) + b.abs()
                if l < 4:
                    x = torch.relu(x)
                if l in (2, 3):
                    g, be, mu, var = (self.t64(c) for c in self.bn_raw[l - 2])
                    sc = g / torch.sqrt(var + 1e-3)
                    x, m = (x - mu) * sc + be, sc.abs() * m + (be - mu * sc).abs()
                out[l] = (x, m)
        return out


# ---- the per-layer check -----------------------------------------------------------------------------------------
def _where(l, flat_idx, per):
    """'row r (d, h, w, c) = ...' of a flat index into a layer of `per` values per row."""
    r, i = divmod(int(flat_idx), per)
    if l <= 2:
        pos, ch = divmod(i, {0: 5, 1: 16, 2: 32}[l])
        return "row %d (d, h, w, c) = (%d, %d, %d, %d)" % (r, pos // 64, pos // 8 % 8, pos % 8, ch)
    return "row %d column %d" % (r, i)


def _ratios(got, ref, mag, allow):
    err = torch.clamp((got - ref).abs() - allow, min=0)
    return torch.where(err == 0, torch.zeros_like(err), err / torch.clamp(mag, min=1e-300))


def check_rms(l, got, ref, mag, tau_rms, what, tag="", allow=0.0):
    """Root mean square of (|got - ref| - allow) / M over a layer; raises when it passes tau_rms.  A product left out
    of one K block or one tap moves every output a little, where the accumulator's rounding only shows in the tail:
    the mean sees the first far below the worst case of the second."""
    r = _ratios(got, ref, mag, allow)
    rms = float(torch.sqrt((r * r).mean())) if r.numel() else 0.0
    if not rms <= tau_rms:
        raise AssertionError("%s%s: rms of |kernel - %s| / M = 2^%.2f > 2^%.2f" % (
            tag, LAYER_NAMES[l], what, np.log2(rms), np.log2(tau_rms)))
    return rms


def check_bound(l, got, ref, mag, tau, what, tag="", allow=0.0):
    """Worst (|got - ref| - allow) / M over a layer (tensors (n, per)); raises naming the layer and the worst element
    when it passes tau."""
    r = _ratios(got, ref, mag, allow)
    if r.numel() == 0:
        return 0.0
    k = int(torch.argmax(r.reshape(-1)))
    worst = float(r.reshape(-1)[k])
    if not worst <= tau:
        raise AssertionError("%s%s: |kernel - %s| / M = 2^%.2f > tau = 2^%.2f at %s: kernel %.9g, %s %.9g, M %.3g" % (
            tag, LAYER_NAMES[l], what, np.log2(worst), np.log2(tau), _where(l, k, r.shape[1]),
            float(got.reshape(-1)[k]), what, float(ref.reshape(-1)[k]), float(mag.reshape(-1)[k])))
    return worst


def check_layers(net, feats, outs, tau, tau_exact, tau_rms, tag="", layers=(0, 1, 2, 3, 4)):
    """Checks the kernel outputs of one run layer by layer.  outs[l] = (hi, lo) uint16 bits of shape (n, per) for
    l = 0..3 (numpy or torch), outs[4] = fp32 keypoints (n, 57).  feats: the fp32 feature maps of the run's rows, in
    the run's order.  Layer l > 0 is checked against the references evaluated from outs[l - 1]; tau, tau_exact and
    tau_rms are {layer: bound}.  Returns {layer: (worst ratio against the emulation, worst ratio against exact float64,
    rms ratio against the emulation)}."""
    n, dev = len(feats), net.device
    shapes = {0: (n, net.D, 8, 8, 5), 1: (n, net.D, 8, 8, 16), 2: (n, -1), 3: (n, -1)}
    bits = {l: tuple(_t(p, dev) for p in outs[l]) for l in range(4) if l in outs}
    stats = {}
    if 0 in layers:
        hi, lo = split(_t(np.asarray(feats, np.float32).reshape(n, -1), dev))
        bad = (bits[0][0] != hi) | (bits[0][1] != lo)
        if bool(bad.any()):
            k = int(torch.argmax(bad.reshape(-1).to(torch.int8)))
            raise AssertionError("%s%s: not the bf16 split of the feature maps at %s" % (
                tag, LAYER_NAMES[0], _where(0, k, bad.shape[1])))
        stats[0] = (0.0, 0.0, 0.0)
    for l in (1, 2, 3, 4):
        if l not in layers:
            continue
        ph, pl = bits[l - 1]
        a_hi, a_lo = bf16_value(ph).reshape(shapes[l - 1]), bf16_value(pl).reshape(shapes[l - 1])
        emu, exact, mag = (x.reshape(n, -1) for x in net.layer(l, a_hi, a_lo))
        if l == 4:
            got, allow = net.t64(np.asarray(outs[4], np.float32)).reshape(n, -1), 0.0
        else:
            hi, lo = bits[l]
            bad = split_violations(hi, lo)
            if bool(bad.any()):
                k = int(torch.argmax(bad.reshape(-1).to(torch.int8)))
                raise AssertionError("%s%s: (hi, lo) = (0x%04x, 0x%04x) is not a round-to-nearest split at %s" % (
                    tag, LAYER_NAMES[l], int(hi.reshape(-1)[k]) & 0xFFFF, int(lo.reshape(-1)[k]) & 0xFFFF,
                    _where(l, k, hi.shape[1])))
            got, allow = decode(hi, lo), split_allowance(hi, lo)
        stats[l] = (check_bound(l, got, emu, mag, tau[l], "emulation", tag, allow),
                    check_bound(l, got, exact, mag, tau_exact[l], "exact float64", tag, allow),
                    check_rms(l, got, emu, mag, tau_rms[l], "emulation", tag, allow))
    return stats


# ---- an emulated build on the CPU (fp32 accumulation), for the checker's self-test -----------------------------------
MUTATIONS = {
    "conv2_tap_alo": 2,        # conv 2 tap 13 (of 27) without its a_lo w_hi product
    "dense1_kblock_alo": 3,    # dense 1 K block 37 (of 96) without its a_lo w_hi product
    "trunc_split": 1,          # every epilogue splits by truncation instead of round-to-nearest
    "bn1_shift": 2,            # BN 1 channel 5's shift off by 1e-3
}


def emulated_build(net, feats, mutation=None):
    """The outputs check_layers takes, computed the way the kernels compute them but with torch fp32 convolutions and
    matrix products on the CPU; mutation: None (correct) or a key of MUTATIONS."""
    n, D = len(feats), net.D
    f32 = lambda a: _t(a, "cpu", torch.float32)
    sp = split_trunc if mutation == "trunc_split" else split
    outs = {0: split(f32(np.asarray(feats, np.float32).reshape(n, -1)))}
    pad = (1, 1, 1) if D == 3 else (0, 1, 1)
    conv32 = lambda x, k: Fn.conv3d(x.permute(0, 4, 1, 2, 3), k.permute(4, 3, 0, 1, 2), padding=pad).permute(0, 2, 3, 4, 1)
    with torch.no_grad():
        for l in (1, 2, 3, 4):
            shape = (n, D, 8, 8, -1) if l <= 2 else (n, -1)
            a_hi, a_lo = (bf16_value(p).float().reshape(shape) for p in outs[l - 1])
            w = net.k[l - 1] if l <= 2 else net.wd[l - 3]
            wh, wl = (bf16_value(b).float() for b in split(w))
            op = conv32 if l <= 2 else (lambda a, b: a @ b)
            wh_for_lo = wh
            if mutation == "conv2_tap_alo" and l == 2:
                wh_for_lo = wh.clone()
                wh_for_lo.reshape(-1, *wh.shape[3:])[13] = 0
            if mutation == "dense1_kblock_alo" and l == 3:
                a_lo = a_lo.clone()
                a_lo[:, 37 * 64:38 * 64] = 0
            v = op(a_hi, wh) + op(a_lo, wh_for_lo) + op(a_hi, wl) + f32(net.b[l - 1])
            if l == 4:
                outs[4] = v.reshape(n, -1).numpy()
                break
            v = torch.relu(v)
            if l >= 2:
                s, t = net.bn_f32[l - 2]
                if mutation == "bn1_shift" and l == 2:
                    t = t.copy()
                    t[5] += np.float32(1e-3)
                v = (v.double() * _t(s).double() + _t(t).double()).float()      # fmaf: one rounding
            outs[l] = sp(v.reshape(n, -1))
    return outs

"""Training input pipeline of auto_pose/ae/dataset.py:456-495 (``Dataset.batch``) with the image work on the GPU: background
paste by mask + the imgaug chain the training cfg names under ``[Augmentation] CODE`` (auto_pose/ae/cfg/train_template.cfg:26-37).

The cfg string is evaluated against recording stand-ins for the imgaug classes (imgaug itself is not needed), the per-image
random draws are made here with numpy (same distributions as imgaug's stochastic parameters, not its random stream), and
``aae_augment_batch`` applies them: cv2.warpAffine / cv2.GaussianBlur / cv2.resize(NEAREST) arithmetic bit for bit, the
value ops as composed 256-entry tables (include/aae_b200.h).  At the tensor-core trainer's ~10 000 images/s the reference's
10 Python threads of imgaug would be the bottleneck by more than an order of magnitude.

Supported chain: any subset of the template's ops IN THE TEMPLATE'S ORDER (Affine, CoarseDropout, GaussianBlur, Add, Invert,
Multiply, Multiply, ContrastNormalization; another order raises): Sometimes(p, Affine(scale=(a, b))), Sometimes(p, CoarseDropout(p=, size_percent=)),
Sometimes(p, GaussianBlur(sigma)), Sometimes(p, Add((a, b), per_channel=)), Sometimes(p, Invert(p, per_channel=True)),
Sometimes(p, Multiply((a, b), per_channel=)), Sometimes(p, ContrastNormalization((a, b), per_channel=)).  Anything else raises.
"""
import ctypes as C

import numpy as np
import torch

from .. import _lib

FLAG_AFFINE, FLAG_DROP, FLAG_BLUR = 1, 2, 4


# ----------------------------------------------------------------------------------------------------------- cfg parsing
class _Op(object):
    def __init__(self, kind, *args, **kw):
        self.kind, self.args, self.kw = kind, args, kw

    def __repr__(self):
        return "%s%r%r" % (self.kind, self.args, self.kw)


def _recorder(kind):
    return lambda *a, **k: _Op(kind, *a, **k)


def parse_code(code):
    """``CODE`` string of the training cfg -> list of (probability, _Op).  ``np`` inside the string is numpy (the template
    draws the blur sigma with np.random.rand() once, when the cfg is evaluated -- as the reference does)."""
    names = ["Affine", "CoarseDropout", "GaussianBlur", "Add", "Invert", "Multiply", "ContrastNormalization", "LinearContrast",
             "PerspectiveTransform", "CropAndPad", "Fliplr", "Flipud", "AdditiveGaussianNoise", "Dropout"]
    ns = {n: _recorder(n) for n in names}
    ns["np"] = np
    ns["Sometimes"] = lambda p, op, *a, **k: (float(p), op)
    ns["Sequential"] = lambda ops, random_order=False, **k: ("seq", list(ops), bool(random_order))
    tag, ops, random_order = eval(code, {"__builtins__": {}}, ns)    # the reference evals the same string against imgaug (dataset.py:60-64)
    if random_order:
        raise NotImplementedError("Sequential(random_order=True) is not supported")
    out = []
    for item in ops:
        p, op = item if isinstance(item, tuple) else (1.0, item)
        if op.kind not in ("Affine", "CoarseDropout", "GaussianBlur", "Add", "Invert", "Multiply", "ContrastNormalization", "LinearContrast"):
            raise NotImplementedError("augmenter %s is not supported on the device pipeline" % op.kind)
        out.append((p, op))
    return out


def _range(v):
    if isinstance(v, (tuple, list)):
        return float(v[0]), float(v[1])
    return float(v), float(v)


# ----------------------------------------------------------------------------------------------------------- OpenCV tables
def bilinear_table():
    """OpenCV's INTER_LINEAR fixed-point weight table (initInterTab2D): [32*32][4] uint16 (the weight of an exact pixel hit is
    32768 itself), every row sums to 32768."""
    t = np.arange(32, dtype=np.float32) / np.float32(32)
    c = np.stack([np.float32(1) - t, t], 1).astype(np.float32)
    w = (c[:, None, :, None] * c[None, :, None, :]).astype(np.float32).reshape(32 * 32, 4)      # [fy][fx][(ky, kx)]
    it = np.rint(w * np.float32(32768)).astype(np.int32)
    for row in it:
        diff = int(row.sum()) - 32768
        if diff:
            mk, big = 0, 0
            for k in range(4):
                if row[k] < row[mk]:
                    mk = k
                elif row[k] > row[big]:
                    big = k
            if diff < 0:
                row[big] -= diff
            else:
                row[mk] -= diff
    return it.astype(np.uint16)


def affine_tables(M, h, w):
    """cv2.warpAffine's fixed-point coordinate tables for the forward matrix M [2,3]: adelta[w], bdelta[w], X0[h], Y0[h] (int32)."""
    M = np.array(M, np.float64).reshape(2, 3).copy()
    D = M[0, 0] * M[1, 1] - M[0, 1] * M[1, 0]
    D = 1.0 / D if D != 0 else 0.0
    a11, a22 = M[1, 1] * D, M[0, 0] * D
    M[0, 0] = a11
    M[0, 1] *= -D
    M[1, 0] *= -D
    M[1, 1] = a22
    b1 = -M[0, 0] * M[0, 2] - M[0, 1] * M[1, 2]
    b2 = -M[1, 0] * M[0, 2] - M[1, 1] * M[1, 2]
    M[0, 2], M[1, 2] = b1, b2
    xs, ys = np.arange(w, dtype=np.float64), np.arange(h, dtype=np.float64)
    adelta = np.rint(M[0, 0] * xs * 1024.0)
    bdelta = np.rint(M[1, 0] * xs * 1024.0)
    X0 = np.rint((M[0, 1] * ys + M[0, 2]) * 1024.0) + 16
    Y0 = np.rint((M[1, 1] * ys + M[1, 2]) * 1024.0) + 16
    return adelta.astype(np.int32), bdelta.astype(np.int32), X0.astype(np.int32), Y0.astype(np.int32)


def gaussian_taps_q8(sigma):
    """OpenCV's fixed-point 5-tap Gaussian (8 fractional bits): outer taps rounded with error diffusion, centre = 256 - 2 * (t0 + t1)."""
    x = np.arange(5, dtype=np.float64) - 2.0
    k = np.exp(-x * x / (2.0 * sigma * sigma))
    k /= k.sum()
    kq = np.zeros(5, np.int32)
    err = 0.0
    for i in range(2):
        adj = k[i] * 256.0 + err
        v0 = int(np.rint(adj))
        err = adj - v0
        kq[i] = kq[4 - i] = v0
    kq[2] = 256 - 2 * int(kq[0] + kq[1])
    return kq


def nearest_cells(dst, src, dtype=np.uint8):
    """cv2.resize INTER_NEAREST: source index of each of the dst output cells for a source of src cells"""
    ifx = 1.0 / (float(dst) / float(src))
    return np.minimum(np.floor(np.arange(dst, dtype=np.float64) * ifx).astype(np.int64), src - 1).astype(dtype)


_IDENT = np.arange(256, dtype=np.uint8)


def _lut_add(v):
    return np.clip(np.arange(256, dtype=np.int16) + int(v), 0, 255).astype(np.uint8)


def _lut_mul(m):
    return np.clip(np.arange(256, dtype=np.float32) * np.float32(m), 0, 255).astype(np.uint8)


def _lut_contrast(a):
    return np.clip(np.float32(127) + np.float32(a) * (np.arange(256, dtype=np.float32) - np.float32(127)), 0, 255).astype(np.uint8)


# ----------------------------------------------------------------------------------------------------------- augmenter
class Augmenter(object):
    def __init__(self, code, shape=(128, 128, 3), seed=None):
        self.h, self.w, self.c = int(shape[0]), int(shape[1]), int(shape[2])
        self.ops = parse_code(code) if isinstance(code, str) else list(code)
        canon = ["Affine", "CoarseDropout", "GaussianBlur", "Add", "Invert", "Multiply", "Multiply", "ContrastNormalization"]
        pos = 0
        for _, op in self.ops:                                  # the kernels apply the ops in the template's order
            kind = "ContrastNormalization" if op.kind == "LinearContrast" else op.kind
            while pos < len(canon) and canon[pos] != kind:
                pos += 1
            if pos == len(canon):
                raise NotImplementedError("augmenter order %s is not a sub-sequence of %s" % ([o.kind for _, o in self.ops], canon))
            pos += 1
        self.rng = np.random.RandomState(seed)
        self.sigma = 0.0
        self.low = (1, 1)
        for _, op in self.ops:
            if op.kind == "GaussianBlur":
                self.sigma = float(op.args[0] if op.args else op.kw.get("sigma", 0.0))
                if self.sigma >= 1.5:
                    raise NotImplementedError("GaussianBlur sigma >= 1.5 needs a kernel larger than 5 taps")
            if op.kind == "CoarseDropout":
                sp = float(op.kw.get("size_percent", 0.05))
                self.low = (max(int(self.h * sp), 4), max(int(self.w * sp), 4))     # FromLowerResolution(min_size=4)
                if self.low[0] * self.low[1] > 64:
                    raise NotImplementedError("CoarseDropout masks with more than 64 cells are not supported")
        self._dev = {}

    # -- host: random draws (imgaug's distributions; numpy's stream) -------------------------------------------------
    def sample(self, B):
        """Per-image parameters of one batch: dict of arrays (``*_on`` = the Sometimes draw, values per image / channel)."""
        r, C_ = self.rng, self.c
        P = {"affine_on": np.zeros(B, bool), "affine_M": np.tile(np.array([[1.0, 0, 0], [0, 1.0, 0]]), (B, 1, 1)),
             "drop_on": np.zeros(B, bool), "drop_keep": np.ones((B,) + self.low, np.uint8), "blur_on": np.zeros(B, bool),
             "add_on": np.zeros(B, bool), "add_val": np.zeros((B, C_), np.int32), "invert_on": np.zeros(B, bool),
             "invert_ch": np.zeros((B, C_), bool), "mul1_on": np.zeros(B, bool), "mul1_val": np.ones((B, C_), np.float32),
             "mul2_on": np.zeros(B, bool), "mul2_val": np.ones((B, C_), np.float32), "contrast_on": np.zeros(B, bool),
             "contrast_val": np.ones((B, C_), np.float32)}
        n_mul = 0

        def per_channel(pc, draw):
            """value per channel: with probability pc (True = 1, False = 0) independent draws, else one draw repeated"""
            v = draw((B, C_))
            same = r.rand(B) >= float(pc)
            v[same] = v[same][:, :1]
            return v

        for p, op in self.ops:
            on = r.rand(B) < p
            if op.kind == "Affine":
                lo, hi = _range(op.kw.get("scale", 1.0))
                s = r.uniform(lo, hi, B)
                cx, cy = self.w / 2.0 - 0.5, self.h / 2.0 - 0.5
                P["affine_on"] = on
                for b in range(B):
                    P["affine_M"][b] = [[s[b], 0.0, cx - s[b] * cx], [0.0, s[b], cy - s[b] * cy]]
            elif op.kind == "CoarseDropout":
                P["drop_on"] = on
                P["drop_keep"] = (r.rand(B, *self.low) >= float(op.kw.get("p", op.args[0] if op.args else 0.0))).astype(np.uint8)
            elif op.kind == "GaussianBlur":
                P["blur_on"] = on
            elif op.kind == "Add":
                lo, hi = _range(op.args[0] if op.args else op.kw.get("value", 0))
                P["add_on"] = on
                P["add_val"] = per_channel(op.kw.get("per_channel", False), lambda sz: r.randint(int(lo), int(hi) + 1, sz)).astype(np.int32)
            elif op.kind == "Invert":
                P["invert_on"] = on
                pi = float(op.args[0] if op.args else op.kw.get("p", 0.0))
                P["invert_ch"] = per_channel(op.kw.get("per_channel", False), lambda sz: (r.rand(*sz) < pi)).astype(bool)
            elif op.kind == "Multiply":
                lo, hi = _range(op.args[0] if op.args else op.kw.get("mul", 1.0))
                key = "mul1" if n_mul == 0 else "mul2"
                if n_mul > 1:
                    raise NotImplementedError("more than two Multiply stages")
                n_mul += 1
                P[key + "_on"] = on
                P[key + "_val"] = per_channel(op.kw.get("per_channel", False), lambda sz: r.uniform(lo, hi, sz)).astype(np.float32)
            else:  # ContrastNormalization / LinearContrast
                lo, hi = _range(op.args[0] if op.args else op.kw.get("alpha", 1.0))
                P["contrast_on"] = on
                P["contrast_val"] = per_channel(op.kw.get("per_channel", False), lambda sz: r.uniform(lo, hi, sz)).astype(np.float32)
        return P

    # -- host: pack the draws into the two device buffers ------------------------------------------------------------
    def pack(self, P):
        """-> geom int32 [B, 4 + 2W + 2H], lut uint8 [B, C, 256] (include/aae_b200.h: aae_augment_batch); vectorised over the batch."""
        B = len(P["affine_on"])
        H, W, C_ = self.h, self.w, self.c
        geom = np.zeros((B, 4 + 2 * W + 2 * H), np.int32)
        blur = bool(self.sigma > 1e-3)
        geom[:, 0] = (P["affine_on"].astype(np.int32) * FLAG_AFFINE) | (P["drop_on"].astype(np.int32) * FLAG_DROP) | \
                     ((P["blur_on"] & blur).astype(np.int32) * FLAG_BLUR)
        weights = (np.uint64(1) << np.arange(self.low[0] * self.low[1], dtype=np.uint64))
        keep = (P["drop_keep"].reshape(B, -1).astype(np.uint64) * weights[None, :]).sum(1, dtype=np.uint64)
        geom[:, 1] = (keep & np.uint64(0xFFFFFFFF)).astype(np.uint32).view(np.int32)
        geom[:, 2] = (keep >> np.uint64(32)).astype(np.uint32).view(np.int32)
        on = np.nonzero(P["affine_on"])[0]
        if len(on):
            # cv2.warpAffine: invert the forward matrix in double, then 10-bit fixed-point column / row tables (affine_tables, batched)
            M = np.array(P["affine_M"][on], np.float64)
            D = M[:, 0, 0] * M[:, 1, 1] - M[:, 0, 1] * M[:, 1, 0]
            D = np.where(D != 0, 1.0 / np.where(D != 0, D, 1.0), 0.0)
            a11, a22 = M[:, 1, 1] * D, M[:, 0, 0] * D
            m01, m10 = M[:, 0, 1] * -D, M[:, 1, 0] * -D
            b1 = -a11 * M[:, 0, 2] - m01 * M[:, 1, 2]
            b2 = -m10 * M[:, 0, 2] - a22 * M[:, 1, 2]
            xs, ys = np.arange(W, dtype=np.float64)[None, :], np.arange(H, dtype=np.float64)[None, :]
            geom[on, 4:4 + W] = np.rint(a11[:, None] * xs * 1024.0).astype(np.int32)
            geom[on, 4 + W:4 + 2 * W] = np.rint(m10[:, None] * xs * 1024.0).astype(np.int32)
            geom[on, 4 + 2 * W:4 + 2 * W + H] = (np.rint((m01[:, None] * ys + b1[:, None]) * 1024.0) + 16).astype(np.int32)
            geom[on, 4 + 2 * W + H:] = (np.rint((a22[:, None] * ys + b2[:, None]) * 1024.0) + 16).astype(np.int32)
        # value ops: one uint8 -> uint8 table per (image, channel) = the op chain evaluated on the 256 possible values, every op
        # with the arithmetic of its imgaug uint8 table (integer add + clip; float32 multiply, clip, truncate)
        t = np.broadcast_to(np.arange(256, dtype=np.int32)[None, None, :], (B, C_, 256))
        f127 = np.float32(127)

        def sel(on_b, new):
            m = on_b[:, None, None] if on_b.ndim == 1 else on_b[:, :, None]
            return np.where(m, new, t)

        if P["add_on"].any():
            t = sel(P["add_on"], np.clip(t + P["add_val"].astype(np.int32)[:, :, None], 0, 255))
        inv = P["invert_on"][:, None] & P["invert_ch"]
        if inv.any():
            t = sel(inv, 255 - t)
        for key in ("mul1", "mul2"):
            if P[key + "_on"].any():
                t = sel(P[key + "_on"], np.clip(t.astype(np.float32) * P[key + "_val"].astype(np.float32)[:, :, None], 0, 255).astype(np.uint8).astype(np.int32))
        if P["contrast_on"].any():
            c = f127 + P["contrast_val"].astype(np.float32)[:, :, None] * (t.astype(np.float32) - f127)
            t = sel(P["contrast_on"], np.clip(c, 0, 255).astype(np.uint8).astype(np.int32))
        # t may still be the stride-0 broadcast view (no value op fired): astype would keep a permuted memory order, and the
        # kernel reads raw [B][C][256] memory
        return np.ascontiguousarray(geom), np.ascontiguousarray(t, dtype=np.uint8)

    # -- device ------------------------------------------------------------------------------------------------------
    def _constants(self, dev):
        key = str(dev)
        if key not in self._dev:
            self._dev[key] = {
                "tab": torch.from_numpy(bilinear_table().view(np.int16)).to(dev),     # raw 16-bit patterns (torch has no uint16 arithmetic)
                "rows": torch.from_numpy(nearest_cells(self.h, self.low[0])).to(dev),
                "cols": torch.from_numpy(nearest_cells(self.w, self.low[1])).to(dev),
                "to_float": torch.from_numpy((np.arange(256) / 255.).astype(np.float32)).to(dev),     # batch_x / 255. then the float32 feed
                "taps": gaussian_taps_q8(self.sigma).astype(np.int32) if self.sigma > 1e-3 else None,
            }
        return self._dev[key]

    def augment_device(self, x, mask, bg, params=None, want_u8=False):
        """x, bg: uint8 CUDA tensors [B,H,W,C]; mask: bool/uint8 CUDA tensor [B,H,W] (True = background).  Returns the float32
        batch in [0, 1] the training step consumes (and the uint8 image when want_u8)."""
        dev = x.device
        B = x.shape[0]
        P = params if params is not None else self.sample(B)
        geom, lut = self.pack(P)
        geom, lut = np.ascontiguousarray(geom, dtype=np.int32), np.ascontiguousarray(lut, dtype=np.uint8)
        if geom.shape != (B, 4 + 2 * self.w + 2 * self.h) or lut.shape != (B, self.c, 256):
            raise ValueError("augmentation tables have shapes %s / %s for a batch of %d" % (geom.shape, lut.shape, B))
        k = self._constants(dev)
        geom_d, lut_d = torch.from_numpy(geom).to(dev, non_blocking=True), torch.from_numpy(lut).to(dev, non_blocking=True)
        assert geom_d.is_contiguous() and lut_d.is_contiguous()
        mask8 = mask.to(torch.uint8).contiguous()
        tmp = torch.empty_like(x)
        out_f = torch.empty(x.shape, dtype=torch.float32, device=dev)
        out_u = torch.empty_like(x) if want_u8 else None
        taps = k["taps"]
        _lib.check(_lib.lib().aae_augment_batch(_lib.ptr(x.contiguous()), _lib.ptr(mask8), _lib.ptr(bg.contiguous()), B, self.h, self.w, self.c,
                                                _lib.ptr(geom_d), _lib.ptr(lut_d), _lib.ptr(k["tab"]), _lib.ptr(k["rows"]), _lib.ptr(k["cols"]),
                                                self.low[1], _lib.ptr(taps) if taps is not None else None, _lib.ptr(k["to_float"]), _lib.ptr(tmp),
                                                _lib.ptr(out_u) if out_u is not None else None, _lib.ptr(out_f),
                                                C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)), "augment batch")
        return (out_f, out_u) if want_u8 else out_f

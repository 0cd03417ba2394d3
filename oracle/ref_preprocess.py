"""TEST INFRASTRUCTURE ONLY - CPU restatement of the reference's image pre-processing (SURVEY.md 8f row 3).

`load_and_preprocess` follows iggt/utils/load_fn.py:12-128 step by step.  The resize itself lives in a third-party
dependency of the reference, Pillow (`img.resize(size, Image.Resampling.BICUBIC)`, load_fn.py:82; Pillow 12.2.0 in this
image): `resize_bicubic_u8` restates its published 8-bit algorithm (src/libImaging/Resample.c: bicubic_filter,
precompute_coeffs, normalize_coeffs_8bpc, ImagingResampleHorizontal_8bpc / Vertical_8bpc) with scalar Python loops for
the taps and integer numpy for the accumulation.  Pinned by tests/test_preprocess.py against Pillow itself and against
tests/golden/preprocess_ref.json, which oracle/make_golden_preprocess.py produced by running the unmodified reference
function.  Nothing outside tests/, smoke() and bench.py's CPU legs may import this module."""
import math

import numpy as np

PRECISION_BITS = 32 - 8 - 2


def bicubic_filter(x: float) -> float:
    a = -0.5
    if x < 0.0:
        x = -x
    if x < 1.0:
        return ((a + 2.0) * x - (a + 3.0)) * x * x + 1
    if x < 2.0:
        return (((x - 5) * x + 8) * x - 4) * a
    return 0.0


def precompute_coeffs(in_size: int, out_size: int):
    """Returns (ksize, bounds[(xmin, xmax)], taps as Python ints) for one pass over the full axis (box = whole image)."""
    scale = filterscale = float(in_size) / out_size
    if filterscale < 1.0:
        filterscale = 1.0
    support = 2.0 * filterscale
    ksize = int(math.ceil(support)) * 2 + 1
    bounds, taps = [], []
    ss = 1.0 / filterscale
    for xx in range(out_size):
        center = 0.0 + (xx + 0.5) * scale
        xmin = int(center - support + 0.5)          # C (int) cast: truncation toward zero
        if xmin < 0:
            xmin = 0
        xmax = int(center + support + 0.5)
        if xmax > in_size:
            xmax = in_size
        xmax -= xmin
        k, ww = [], 0.0
        for x in range(xmax):
            w = bicubic_filter((x + xmin - center + 0.5) * ss)
            k.append(w)
            ww += w
        if ww != 0.0:
            k = [w / ww for w in k]
        fixed = [int(-0.5 + w * (1 << PRECISION_BITS)) if w < 0 else int(0.5 + w * (1 << PRECISION_BITS)) for w in k]
        bounds.append((xmin, xmax))
        taps.append(fixed)
    return ksize, bounds, taps


def _pass(img: np.ndarray, out_size: int, axis: int) -> np.ndarray:
    """One 8-bit resampling pass along `axis` of a [H, W, C] uint8 image."""
    src = np.moveaxis(img, axis, 0).astype(np.int64)
    _, bounds, taps = precompute_coeffs(src.shape[0], out_size)
    out = np.empty((out_size,) + src.shape[1:], dtype=np.uint8)
    for xx, ((xmin, xmax), k) in enumerate(zip(bounds, taps)):
        acc = np.full(src.shape[1:], 1 << (PRECISION_BITS - 1), dtype=np.int64)
        for x in range(xmax):
            acc += src[xmin + x] * k[x]
        out[xx] = np.clip(acc >> PRECISION_BITS, 0, 255).astype(np.uint8)
    return np.moveaxis(out, 0, axis)


def resize_bicubic_u8(img: np.ndarray, new_width: int, new_height: int) -> np.ndarray:
    """uint8 [H, W, 3] -> uint8 [new_height, new_width, 3]: horizontal pass, u8 intermediate, vertical pass."""
    h, w = img.shape[:2]
    if (w, h) == (new_width, new_height):
        return img.copy()
    out = img
    if w != new_width:
        out = _pass(out, new_width, 1)
    if h != new_height:
        out = _pass(out, new_height, 0)
    return out


def load_and_preprocess(frames, mode="crop", resize_target_size=None) -> np.ndarray:
    """frames: decoded RGB uint8 [H, W, 3] arrays.  Returns float32 [N, 3, H', W'] like load_fn.py:12-128."""
    target = 518
    outs = []
    for f in frames:
        height, width = f.shape[:2]
        if mode == "pad":
            if width >= height:
                new_w, new_h = target, round(height * (target / width) / 14) * 14
            else:
                new_h, new_w = target, round(width * (target / height) / 14) * 14
        elif mode == "resize":
            new_w, new_h = resize_target_size
        else:
            new_w, new_h = target, round(height * (target / width) / 14) * 14
        img = resize_bicubic_u8(f, new_w, new_h).astype(np.float32).transpose(2, 0, 1) / np.float32(255)
        if mode == "crop" and new_h > target:
            y0 = (new_h - target) // 2
            img = img[:, y0:y0 + target]
        elif mode == "pad":
            hp, wp = target - img.shape[1], target - img.shape[2]
            if hp > 0 or wp > 0:
                img = np.pad(img, ((0, 0), (hp // 2, hp - hp // 2), (wp // 2, wp - wp // 2)), constant_values=1.0)
        outs.append(img)
    mh, mw = max(o.shape[1] for o in outs), max(o.shape[2] for o in outs)
    res = []
    for o in outs:
        hp, wp = mh - o.shape[1], mw - o.shape[2]
        if hp > 0 or wp > 0:
            o = np.pad(o, ((0, 0), (hp // 2, hp - hp // 2), (wp // 2, wp - wp // 2)), constant_values=1.0)
        res.append(o)
    return np.stack(res).astype(np.float32)

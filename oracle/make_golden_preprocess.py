"""Generates tests/golden/preprocess/*.png and tests/golden/preprocess_ref.json by running the UNMODIFIED reference
`iggt.utils.load_fn.load_and_preprocess_images` (it only needs torch, Pillow and torchvision, all present here) on
small synthetic views.  Each output is recorded as its shape and the SHA-256 of round(x * 255) in uint8 (ToTensor's
x / 255 is exactly invertible, so the digest pins every value bit for bit; the arrays themselves run to megabytes).

    python oracle/make_golden_preprocess.py        # needs /root/reference; the fixtures are committed
"""
import hashlib
import importlib.util
import json
import os
import sys

import numpy as np
from PIL import Image

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "tests", "golden", "preprocess")


def synthetic(h, w, seed, alpha=False):
    """Smooth colour gradients + hard-edged boxes + a little noise: exercises overshoot clamping and every tap."""
    g = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float64)
    img = np.stack([127 + 120 * np.sin(xx / (7 + seed) + yy / 13), 255 * xx / w, 255 * (yy / h) ** 2], -1)
    for _ in range(12):
        y0, x0 = int(g.integers(0, h - 4)), int(g.integers(0, w - 4))
        img[y0:y0 + int(g.integers(2, h // 3)), x0:x0 + int(g.integers(2, w // 3))] = g.integers(0, 256, 3)
    img = np.clip(img + g.integers(-6, 7, img.shape), 0, 255).astype(np.uint8)
    if alpha:
        a = (255 * (0.5 + 0.5 * np.cos(xx / 9) * np.sin(yy / 5))).astype(np.uint8)
        img = np.concatenate([img, a[..., None]], -1)
    return img


CASES = {                      # name -> (mode, resize_target_size, [(file, h, w, seed, alpha)])
    "crop_landscape": ("crop", None, [("a.png", 120, 213, 1, False), ("b.png", 120, 213, 2, False)]),
    "crop_portrait_ragged": ("crop", None, [("c.png", 260, 173, 3, False), ("d.png", 97, 131, 4, True)]),
    "pad_mixed": ("pad", None, [("e.png", 150, 100, 5, False), ("f.png", 64, 200, 6, False)]),
    "resize_down_up": ("resize", (70, 56), [("g.png", 333, 500, 7, False), ("h.png", 40, 30, 8, False)]),
}


def main():
    spec = importlib.util.spec_from_file_location("ref_load_fn", "/root/reference/iggt/utils/load_fn.py")
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    os.makedirs(OUT, exist_ok=True)
    digests = {}
    for name, (mode, size, files) in CASES.items():
        paths = []
        for fn, h, w, seed, alpha in files:
            p = os.path.join(OUT, fn)
            Image.fromarray(synthetic(h, w, seed, alpha)).save(p, optimize=True)
            paths.append(p)
        out = ref.load_and_preprocess_images(paths, mode=mode, resize_target_size=size)
        q = (out * 255).round().to(dtype=__import__("torch").uint8)
        assert (q.float().div(255) == out).all()
        digests[name] = digest_u8(q.numpy())
        print(name, tuple(out.shape))
    with open(os.path.join(ROOT, "tests", "golden", "preprocess_ref.json"), "w") as f:
        json.dump(digests, f, indent=1)


def digest_u8(q):
    """shape and SHA-256 of a C-ordered uint8 array"""
    assert q.dtype == np.uint8, q.dtype
    return {"shape": list(q.shape), "sha256_u8": hashlib.sha256(np.ascontiguousarray(q).tobytes()).hexdigest()}


if __name__ == "__main__":
    sys.exit(main())

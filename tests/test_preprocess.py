"""Image pre-processing (SURVEY.md 8f row 3): Pillow-exact bicubic resize + ToTensor + crop / pad on the device.

CPU: the oracle restatement is pinned against Pillow itself and against fixtures made by the unmodified reference
`load_and_preprocess_images` (oracle/make_golden_preprocess.py); the product's host-side tap tables are checked against
the oracle's.  GPU: the C-ABI kernels must reproduce the fixtures BIT-EXACTLY (byte / integer work)."""
import glob
import json
import os
import sys

import numpy as np
import pytest
import torch
from PIL import Image

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_preprocess as R                                      # noqa: E402
from oracle.make_golden_preprocess import CASES, digest_u8, synthetic       # noqa: E402
from iggt_official_b200.utils import load_fn                                # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
RAGGED = [(37, 53, 14, 28), (120, 213, 518, 294), (64, 64, 64, 64), (50, 20, 20, 50), (9, 300, 301, 7),
          (200, 3, 5, 70), (1, 1, 4, 4), (33, 47, 47, 33)]              # (h, w, new_w, new_h)


def _assert_equals_reference_fixture(x, name):
    """x (float32 ndarray) equals the reference's output bit for bit: every value is some k / 255 exactly, and the
    bytes k have the reference's shape and SHA-256."""
    q = np.rint(x * np.float32(255)).astype(np.uint8)
    assert np.array_equal(q.astype(np.float32) / np.float32(255), x)
    assert digest_u8(q) == json.load(open(os.path.join(GOLD, "preprocess_ref.json")))[name]


def _decode(path):
    img = Image.open(path)
    if img.mode == "RGBA":
        img = Image.alpha_composite(Image.new("RGBA", img.size, (255, 255, 255, 255)), img)
    return np.asarray(img.convert("RGB"))


@pytest.mark.parametrize("h,w,nw,nh", RAGGED)
def test_oracle_resize_matches_pillow(h, w, nw, nh):
    img = synthetic(max(h, 12), max(w, 12), h + w)[:h, :w]
    want = np.asarray(Image.fromarray(img).resize((nw, nh), Image.Resampling.BICUBIC))
    assert np.array_equal(R.resize_bicubic_u8(img, nw, nh), want)


@pytest.mark.parametrize("name", sorted(CASES))
def test_oracle_matches_reference_fixture(name):
    mode, size, files = CASES[name]
    got = R.load_and_preprocess([_decode(os.path.join(GOLD, "preprocess", f[0])) for f in files], mode, size)
    assert got.dtype == np.float32
    _assert_equals_reference_fixture(got, name)


@pytest.mark.parametrize("n_in,n_out", [(213, 518), (120, 294), (500, 70), (30, 70), (64, 64), (1, 4), (4000, 518), (7, 3)])
def test_host_tap_tables_match_oracle(n_in, n_out):
    kk, bounds = load_fn.precompute_coeffs(n_in, n_out)
    ksize, b_ref, taps = R.precompute_coeffs(n_in, n_out)
    assert kk.shape == (n_out, ksize) and kk.dtype == np.int32
    assert bounds.tolist() == [list(b) for b in b_ref]
    for xx, k in enumerate(taps):
        assert kk[xx, :len(k)].tolist() == k and not kk[xx, len(k):].any()


def test_to_tensor_division_is_ieee():
    """The kernel computes float(v) / 255.0f with IEEE division; torchvision's ToTensor must agree for every byte."""
    v = torch.arange(256, dtype=torch.uint8)
    assert np.array_equal(v.float().div(255).numpy(), np.arange(256, dtype=np.float32) / np.float32(255))


def test_argument_errors_match_reference():
    with pytest.raises(ValueError, match="At least 1 image"):
        load_fn.load_and_preprocess_images([])
    with pytest.raises(ValueError, match="Mode must be"):
        load_fn.load_and_preprocess_images(["x.png"], mode="stretch")
    with pytest.raises(ValueError, match="resize_target_size must be provided"):
        load_fn.preprocess_decoded([np.zeros((4, 4, 3), np.uint8)], mode="resize")
    with pytest.raises(ValueError, match="tuple or list of two"):
        load_fn.preprocess_decoded([np.zeros((4, 4, 3), np.uint8)], mode="resize", resize_target_size=(1, 2, 3))


# ------------------------------------------------------------------------------------------------ GPU

@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_device_matches_reference_fixture(name):
    mode, size, files = CASES[name]
    out = load_fn.load_and_preprocess_images([os.path.join(GOLD, "preprocess", f[0]) for f in files], mode=mode,
                                             resize_target_size=size)
    assert out.is_cuda and out.dtype == torch.float32
    _assert_equals_reference_fixture(out.cpu().numpy(), name)


@pytest.mark.gpu
@pytest.mark.parametrize("h,w,nw,nh", RAGGED + [(1080, 1920, 518, 294), (3000, 4000, 518, 392)])
def test_device_resize_matches_pillow(h, w, nw, nh):
    img = synthetic(max(h, 12), max(w, 12), h + w)[:h, :w]
    want = np.asarray(Image.fromarray(img).resize((nw, nh), Image.Resampling.BICUBIC))
    out = load_fn.preprocess_decoded([img], mode="resize", resize_target_size=(nw, nh))
    got = (out[0] * 255).round().to(torch.uint8).permute(1, 2, 0).cpu().numpy()
    assert np.array_equal(got, want)
    assert torch.equal(out[0].cpu(), torch.from_numpy(want).permute(2, 0, 1).float().div(255))


@pytest.mark.gpu
def test_device_full_size_crop_properties():
    """Full-size views (BASELINE C2: 518 wide): crop window == the same rows of the uncropped resize; flat images stay flat."""
    img = synthetic(1400, 1000, 11)                                    # portrait -> new_h = 728 > 518: centre crop
    crop = load_fn.preprocess_decoded([img], mode="crop")
    full = load_fn.preprocess_decoded([img], mode="resize", resize_target_size=(518, 728))
    assert tuple(crop.shape) == (1, 3, 518, 518)
    assert torch.equal(crop, full[:, :, 105:105 + 518])
    flat = np.full((700, 900, 3), 200, np.uint8)
    out = load_fn.preprocess_decoded([flat], mode="pad")
    body = out[0, :, 58:58 + 403]                                       # 518 x round(700 * 518 / 900 / 14) * 14 = 406
    assert tuple(out.shape) == (1, 3, 518, 518) and float(out.max()) == 1.0
    assert torch.all(body == torch.tensor(200, dtype=torch.float32).div(255))

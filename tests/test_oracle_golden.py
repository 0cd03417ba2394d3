"""CPU: pins the oracle restatement (oracle/ref_model.py) to outputs of the UNMODIFIED reference, generated
by oracle/make_golden.py (which imports /root/reference) and committed under tests/golden/."""
import glob
import os

import pytest
import torch

from oracle import ref_model, weights

GOLDEN = sorted(p for p in glob.glob(os.path.join(os.path.dirname(__file__), "golden", "*.pt"))
                if os.path.basename(p).startswith(("iggt_", "vggt_")))      # the whole-forward fixtures (make_golden.py)
PREFIXES = ("aggregator.", "camera_head.", "depth_head.", "point_head.", "part_adaptor.", "part_head.")


def _rel(a, b):
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-12)).item()


def test_golden_present():
    assert len(GOLDEN) >= 4


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-3] for p in GOLDEN])
def test_oracle_matches_reference(path):
    rec = torch.load(path)
    c = rec["case"]
    sd = weights.make_state_dict(c["wseed"], c["kind"], prefixes=PREFIXES)
    g = torch.Generator().manual_seed(c["iseed"])
    images = torch.rand(c["B"], c["S"], 3, c["H"], c["W"], generator=g)
    toks = ref_model.aggregator(sd, images)
    rows = rec.get("token_rows")           # a seeded sample of the B*S*T token rows, in fixtures of many views
    for i in (4, 23):
        got = toks[i] if rows is None else toks[i].flatten(0, -2)[rows]
        # fp32 vs fp32, different op order only: 5e-5 of the tensor's max magnitude
        assert got.shape == rec[f"tokens{i}"].shape
        assert _rel(got, rec[f"tokens{i}"]) < 5e-5
    out = ref_model.forward(sd, images, model="iggt" if c["model"] == "IGGT" else "vggt", frames_chunk=2)
    pose = torch.stack(out["pose_enc"], 0)
    assert _rel(pose, rec["pose_enc"]) < 1e-4
    keys = ["depth", "depth_conf", "world_points", "world_points_conf"]
    if c["model"] == "IGGT":
        keys.append("part_feat")
    else:
        assert "part_feat" not in out
    for k in keys:
        assert out[k].shape == rec[k].shape, k
        # fp32 restatement vs fp32 reference: only op-order noise is allowed (measured ~2e-6)
        assert _rel(out[k], rec[k]) < 2e-5, k


def test_rpi_buffers_and_manifest():
    man = weights.load_manifest()
    assert len(man) == 2053 and sum(torch.Size(s).numel() for _, s, _ in man) == 1299499573
    assert ref_model.calculate_rpi_sa(8).shape == (64, 64)
    oca = ref_model.calculate_rpi_oca(8)
    # the reference's buffer really holds negative entries (python-style wrap into the 361-row table)
    assert oca.shape == (64, 144) and int(oca.min()) == -200 and int(oca.max()) == 160


def test_part_head_rejects_odd_grid():
    # reference: RuntimeError from window_partition's view on a 37x37 grid (SURVEY F2)
    with pytest.raises(RuntimeError):
        ref_model.part_head({}, [torch.zeros(1, 256, 12, 12)] * 4, None, 42, 42)

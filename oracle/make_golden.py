"""Generates tests/golden/*.pt by running the UNMODIFIED reference (imported from /root/reference with the
shims in oracle/shims.py) on seeded inputs and the synthetic checkpoints of oracle/weights.py.

Run here only (the GPU box has no /root/reference):   python oracle/make_golden.py
The fixtures pin oracle/ref_model.py (tests/test_oracle_golden.py); the reference itself ships no tests or
golden vectors for this path (SURVEY.md section 4), so these are "outputs of the reference itself run here".
"""
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import shims, weights  # noqa: E402

CASES = [
    # name, model class, B, S, H, W, weight kind, weight seed, input seed
    ("iggt_s2_28x56_stress", "IGGT", 1, 2, 28, 56, "stress", 1, 11),
    ("iggt_b2s3_28x28_default", "IGGT", 2, 3, 28, 28, "default", 0, 12),
    ("vggt_s2_42x42_stress", "VGGT", 1, 2, 42, 42, "stress", 2, 13),
    ("iggt_s1_56x84_stress", "IGGT", 1, 1, 56, 84, "stress", 3, 14),
]
# tokens4 / tokens23 are [B, S, T, 2048] fp32; beyond this many B*S*T rows a fixture keeps a seeded sample of rows
# (`token_rows`, indices into the flattened rows) so that it stays under 1 MB.  The prediction heads are kept whole.
MAX_TOKEN_ROWS = 32


def token_rows(n, seed):
    if n <= MAX_TOKEN_ROWS:
        return None
    return torch.randperm(n, generator=torch.Generator().manual_seed(seed))[:MAX_TOKEN_ROWS].sort().values


def main():
    shims.install()
    from iggt.models.vggt import IGGT, VGGT
    os.makedirs(os.path.join(ROOT, "tests", "golden"), exist_ok=True)
    torch.set_grad_enabled(False)
    model = {"IGGT": None, "VGGT": None}
    for name, cls, B, S, H, W, kind, wseed, iseed in CASES:
        t0 = time.time()
        if model[cls] is None:
            model[cls] = (IGGT if cls == "IGGT" else VGGT)().eval()
        m = model[cls]
        sd = weights.make_state_dict(wseed, kind)
        ref_sd = m.state_dict()
        for k in ref_sd:
            if "relative_position_index" in k:
                assert torch.equal(ref_sd[k], sd[k]), k   # restated index buffers are exact
        missing, unexpected = m.load_state_dict(sd, strict=False)
        assert not missing, missing
        if cls == "IGGT":
            assert not unexpected, unexpected
        g = torch.Generator().manual_seed(iseed)
        images = torch.rand(B, S, 3, H, W, generator=g)
        toks = {}
        hook = m.aggregator.register_forward_hook(lambda mod, inp, out: toks.update(
            {i: out[0][i].clone() for i in (4, 23)}))
        out = m(images if B > 1 else images[0])
        hook.remove()
        rec = {"case": dict(name=name, model=cls, B=B, S=S, H=H, W=W, kind=kind, wseed=wseed, iseed=iseed),
               "tokens4": toks[4], "tokens23": toks[23]}
        rows = token_rows(toks[4][..., 0].numel(), iseed)
        if rows is not None:
            rec["token_rows"] = rows
            for i in (4, 23):
                rec[f"tokens{i}"] = toks[i].flatten(0, -2)[rows].clone()
        for k, v in out.items():
            if k == "images":
                continue
            rec[k] = torch.stack(v, 0) if isinstance(v, list) else v
        path = os.path.join(ROOT, "tests", "golden", name + ".pt")
        torch.save(rec, path)
        print(f"{name}: {[ (k, tuple(v.shape)) for k, v in rec.items() if torch.is_tensor(v)]} "
              f"{os.path.getsize(path) / 1e3:.0f} kB in {time.time() - t0:.1f}s")


if __name__ == "__main__":
    main()

"""Generates tests/golden/amp_block_bf16.pt: the UNMODIFIED reference's transformer block (iggt/layers/block.py) and
patch embedding run under `torch.autocast("cpu", dtype=torch.bfloat16)` in this container, with the (input, output) of
every sub-module recorded.  tests/test_oracle_amp.py replays each stage through oracle/ref_model.py's `amp=` mode and
holds it to (near) bit equality - this pins WHERE the restatement rounds to 16 bit (Linear operands, bias and result;
GELU on the 16-bit fc1 output; fp32 LayerScale / residual; SDPA operands) against real autocast instead of against the
builder's reading of it.  CPU autocast differs from CUDA autocast in one documented place (layer_norm is not on its
fp32 list, so q_norm / k_norm / RoPE stay 16-bit): ref_model.AUTOCAST_DEVICE = "cpu" restates exactly that and is
used by this pin only.  Run here only (the GPU box has no /root/reference):   python oracle/make_golden_amp.py"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_model, shims, weights  # noqa: E402

# one sequence on a 2 x 2 patch grid (9 tokens: both RoPE axes vary) keeps the fixture under 1 MB
CASE = dict(name="amp_block_bf16", kind="stress", wseed=1, iseed=3, block="aggregator.frame_blocks.3.", b=1, gh=2, gw=2,
            dino_block="aggregator.patch_embed.blocks.5.")


KEEP = ("attn.qkv", "attn.q_norm", "attn.k_norm", "attn.rope", "attn.proj", "attn", "ls1", "mlp.fc1", "mlp.act", "mlp.fc2",
        "ls2")
KEEP_DINO = ("attn.qkv", "attn", "mlp.fc1")


def main():
    shims.install()
    from iggt.models.aggregator import Aggregator
    torch.set_grad_enabled(False)
    c = CASE
    sd = weights.make_state_dict(c["wseed"], c["kind"], prefixes=("aggregator.",))
    agg = Aggregator().eval()
    missing, _ = agg.load_state_dict({k[len("aggregator."):]: v for k, v in sd.items()}, strict=False)
    assert not missing, missing
    g = torch.Generator().manual_seed(c["iseed"])
    T = 5 + c["gh"] * c["gw"]
    x = torch.randn(c["b"], T, 1024, generator=g)
    pos = ref_model.positions(c["gh"], c["gw"], "cpu")[None].expand(c["b"], -1, -1).contiguous()
    rec = {"case": c, "x": x, "pos": pos}
    for key, blk, kw in (("frame", agg.frame_blocks[3], dict(pos=pos)), ("dino", agg.patch_embed.blocks[5], {})):
        # The stages' own tensors are recorded, not copies: a stage's input is mostly the previous stage's output (or a
        # view of it), and torch.save stores a shared storage once.  The copies only check that no stage wrote to a
        # recorded tensor in place.
        cap, copies = {}, []
        hooks = []
        for n, mod in blk.named_modules():
            if n:
                def hook(mod, inp, out, n=n):
                    cap.setdefault(n, []).append((inp[0], out))
                    copies.append((inp[0], inp[0].clone(), out, out.clone()))
                hooks.append(mod.register_forward_hook(hook))
        with torch.autocast("cpu", dtype=torch.bfloat16):
            y = blk(x, **kw)
        for h in hooks:
            h.remove()
        assert all(torch.equal(a, a0) and torch.equal(b, b0) for a, a0, b, b0 in copies)
        keep = KEEP if key == "frame" else KEEP_DINO
        rec[key] = {"stages": {n: v for n, v in cap.items() if n in keep}, "y": y}
        print(key, {n: [(tuple(i.shape), str(i.dtype), str(o.dtype)) for i, o in v][:1] for n, v in cap.items()})
    # patch embedding conv (layers/patch_embed.py:25-81) on a normalised image batch
    imgs = torch.randn(2, 3, 28, 42, generator=g)
    with torch.autocast("cpu", dtype=torch.bfloat16):
        pe = agg.patch_embed.patch_embed(imgs)
    rec["patch_embed"] = {"images": imgs, "out": pe}
    path = os.path.join(ROOT, "tests", "golden", c["name"] + ".pt")
    torch.save(rec, path)
    print(path, os.path.getsize(path))


if __name__ == "__main__":
    main()

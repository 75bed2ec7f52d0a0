"""Generate tests/golden/*.npz by running the UNMODIFIED reference (/root/reference/models/latte.py).

TEST INFRASTRUCTURE.  Runs only in the build container (the GPU box has no /root/reference);
its outputs are committed.  Usage:  python oracle/make_golden.py [--xl]

The reference module is loaded by file path (NOT `import models`, whose __init__ pulls diffusers —
SURVEY.md §8c) with `oracle/ref_shim` providing the two timm classes it imports.  Weights and
inputs come from `oracle/latte_oracle.make_weights/make_inputs` (seeded), loaded into the reference
with `load_state_dict(strict=True)` so the key contract (SURVEY.md App. B) is exercised too.
"""
import argparse
import hashlib
import importlib.util
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(HERE, "ref_shim"))

from oracle import golden as G  # noqa: E402
from oracle import latte_oracle as O  # noqa: E402

REF = "/root/reference/models/latte.py"
SUBOPS_SAMPLE = 1 << 15     # elements kept of each (3, 64, 576) sub-op output: four of them whole would pass 1 MB


def load_reference():
    spec = importlib.util.spec_from_file_location("ref_latte", REF)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def build_ref_model(ref, cfg: O.LatteConfig, sd):
    m = ref.Latte(input_size=cfg.input_size, patch_size=cfg.patch_size, in_channels=cfg.in_channels,
                  hidden_size=cfg.hidden_size, depth=cfg.depth, num_heads=cfg.num_heads,
                  mlp_ratio=cfg.mlp_ratio, num_frames=cfg.num_frames,
                  class_dropout_prob=cfg.class_dropout_prob, num_classes=cfg.num_classes,
                  learn_sigma=cfg.learn_sigma, extras=cfg.extras)
    missing, unexpected = m.load_state_dict(sd, strict=True)
    assert not missing and not unexpected
    return m.eval()


def weights_digest(sd) -> str:
    h = hashlib.sha256()
    for k in sorted(sd):
        h.update(k.encode())
        h.update(sd[k].numpy().tobytes())
    return h.hexdigest()


def gen_forward(ref, name, batch, wseed, iseed, out_dir, **cfg_kw):
    cfg = O.make_config(name, **cfg_kw)
    sd = O.make_weights(cfg, wseed)
    x, t, y = O.make_inputs(cfg, batch, iseed)
    m = build_ref_model(ref, cfg, sd)
    with torch.no_grad():
        out = m(x, t, y=y if cfg.extras == 2 else None)
        out_cfg = m.forward_with_cfg(x, t, y=y if cfg.extras == 2 else None, cfg_scale=7.0)
        # reference low-precision noise floors (SURVEY.md §6): fp32 weights under bf16 autocast
        with torch.autocast("cpu", dtype=torch.bfloat16):
            out_bf16 = m(x, t, y=y if cfg.extras == 2 else None).float()
    tag = name.replace("/", "_").replace("-", "_").lower()
    suffix = "" if cfg.extras == 2 else f"_extras{cfg.extras}"
    path = os.path.join(out_dir, f"{tag}{suffix}_b{batch}.npz")
    np.savez(path, **G.pack("out", out.numpy()), out_cfg_half_eps=out_cfg[: batch // 2, :, :4].numpy(),
             ref_bf16_maxabs=np.float32((out_bf16 - out).abs().max().item()),
             t=t.numpy(), y=y.numpy(), x_sum=np.float64(x.double().sum().item()),
             weights_sha256=np.array(weights_digest(sd)),
             meta=np.array(f"{name} batch={batch} wseed={wseed} iseed={iseed} extras={cfg.extras} frames={cfg.num_frames} input={cfg.input_size}"))
    print(f"{path}: out absmax {out.abs().max():.4f} std {out.std():.4f}  ref bf16-autocast dev {float((out_bf16 - out).abs().max()):.3e}")


def gen_subops(ref, out_dir):
    """Sub-op goldens from the reference's own sub-modules (SURVEY.md §8c item 2).  The input `xs` is not stored: the
    test draws it again from `subops_inputs` and checks its sum."""
    cfg = O.make_config("Latte-tiny72/2", input_size=16, num_frames=4)
    sd = O.make_weights(cfg, 7)
    m = build_ref_model(ref, cfg, sd)
    D = cfg.hidden_size
    xs, c = O.subops_inputs(cfg)
    tt = torch.tensor([0, 17, 999])
    with torch.no_grad():
        res = dict(
            xs_sum=np.float64(xs.double().sum().item()), c=c.numpy(), t=tt.numpy(),
            t_emb=m.t_embedder(tt).numpy(),
            t_freq=ref.TimestepEmbedder.timestep_embedding(tt, 256).numpy(),
            **G.pack("block0", m.blocks[0](xs, c).numpy(), SUBOPS_SAMPLE),
            **G.pack("attn0", m.blocks[0].attn(xs).numpy(), SUBOPS_SAMPLE),
            **G.pack("mlp0", m.blocks[0].mlp(xs).numpy(), SUBOPS_SAMPLE),
            final=m.final_layer(xs, c).numpy(),
            **G.pack("modulate", ref.modulate(m.blocks[0].norm1(xs), c, c * 0.5).numpy(), SUBOPS_SAMPLE),
            unpatchify=m.unpatchify(torch.arange(2 * 64 * 32, dtype=torch.float32).reshape(2, 64, 32)).numpy(),
        )
        # fresh reference init tables (not loaded from our state dict) to pin the sin-cos restatement
        fresh = ref.Latte(input_size=16, hidden_size=D, depth=2, num_heads=4, num_frames=4, num_classes=5, extras=2)
        res["fresh_pos_embed"] = fresh.pos_embed.numpy()
        res["fresh_temp_embed"] = fresh.temp_embed.numpy()
        res["fresh_out_absmax"] = np.float32(fresh.eval()(torch.randn(1, 4, 4, 16, 16), torch.tensor([3]), y=torch.tensor([1])).abs().max().item())
    np.savez(os.path.join(out_dir, "subops_tiny72.npz"), **res)
    print("subops_tiny72.npz written; fresh-init output absmax (F5 zero-init trap):", res["fresh_out_absmax"])


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--xl", action="store_true", help="also generate the Latte-XL/2 golden (≈1 min CPU)")
    args = ap.parse_args()
    torch.manual_seed(0)
    out_dir = os.path.join(ROOT, "tests", "golden")
    os.makedirs(out_dir, exist_ok=True)
    ref = load_reference()
    gen_subops(ref, out_dir)
    gen_forward(ref, "Latte-tiny64/2", 2, 11, 12, out_dir, input_size=16, num_frames=8)
    gen_forward(ref, "Latte-tiny72/2", 2, 21, 22, out_dir)
    gen_forward(ref, "Latte-tiny72/2", 4, 31, 32, out_dir, extras=1, input_size=16, num_frames=4)
    gen_forward(ref, "Latte-S/2", 2, 0, 123, out_dir)          # BASELINE config 1
    if args.xl:
        gen_forward(ref, "Latte-XL/2", 2, 0, 123, out_dir)     # BASELINE config 2's model

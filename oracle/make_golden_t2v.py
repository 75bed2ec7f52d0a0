"""Generate tests/golden/t2v_*.npz by running the UNMODIFIED reference /root/reference/models/latte_t2v.py.

TEST INFRASTRUCTURE.  Runs only in the build container (the GPU box has no /root/reference); outputs are committed.
Usage:  python oracle/make_golden_t2v.py [--full]     (--full adds the 28-layer 16x512x512 Latte-1 shape, minutes of CPU)

The reference module is loaded by file path with `oracle/ref_shim` on sys.path, which supplies the `diffusers` names it
imports (latte_t2v.py:9-20).  Executed from the reference file as written: `LatteT2V.forward` (:677-941, incl. the
mask -> bias conversion :740-771), `BasicTransformerBlock_` (:126-396), `AdaLayerNormSingle` (:398-428), `FeedForward`
(:70-123), `get_1d_sincos_temp_embed` (:943-944).  Restated by the shim (diffusers 0.24.0 is not available offline): the
spatial `BasicTransformerBlock`, `Attention`, `PatchEmbed`, `CaptionProjection`, `CombinedTimestepSizeEmbeddings`, `GELU`.
Weights / inputs: `oracle/t2v_oracle.make_weights / make_inputs` (seeded), loaded with `load_state_dict(strict=True)`.
"""
import argparse
import hashlib
import importlib.util
import os
import sys
import time

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(HERE, "ref_shim"))

from oracle import golden as G  # noqa: E402
from oracle import t2v_oracle as T  # noqa: E402

REF = "/root/reference/models/latte_t2v.py"


def load_reference():
    spec = importlib.util.spec_from_file_location("ref_latte_t2v", REF)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def build_ref_model(ref, cfg: T.T2VConfig, sd):
    m = ref.LatteT2V(num_attention_heads=cfg.num_attention_heads, attention_head_dim=cfg.attention_head_dim,
                     in_channels=cfg.in_channels, out_channels=cfg.out_channels, num_layers=cfg.num_layers,
                     patch_size=cfg.patch_size, sample_size=cfg.sample_size, cross_attention_dim=cfg.inner_dim,
                     attention_bias=True, activation_fn="gelu-approximate", norm_type="ada_norm_single",
                     norm_elementwise_affine=False, norm_eps=1e-6, num_embeds_ada_norm=1000,
                     caption_channels=cfg.caption_channels, video_length=cfg.video_length)
    full = dict(sd)
    full["caption_projection.y_embedding"] = m.state_dict()["caption_projection.y_embedding"]   # unused buffer
    missing, unexpected = m.load_state_dict(full, strict=True)
    assert not missing and not unexpected
    return m.eval()


def weights_digest(sd) -> str:
    h = hashlib.sha256()
    for k in sorted(sd):
        h.update(k.encode())
        h.update(sd[k].numpy().tobytes())
    return h.hexdigest()


def make_mask(batch, text_len, valid):
    """(B, L) 0/1 prompt mask with `valid[b]` leading ones (the T5 tokenizer pads at the end, pipeline_latte.py:241-262)."""
    m = torch.zeros(batch, text_len, dtype=torch.int64)
    for b in range(batch):
        m[b, : valid[b % len(valid)]] = 1
    return m


def gen_forward(ref, tag, cfg_kw, batch, text_len, wseed, iseed, out_dir, valid=None, temporal=True, digest=True):
    cfg = T.T2VConfig(**cfg_kw)
    sd = T.make_weights(cfg, wseed)
    x, t, text = T.make_inputs(cfg, batch, text_len, iseed)
    m = build_ref_model(ref, cfg, sd)
    mask = make_mask(batch, text_len, valid) if valid is not None else None
    t0 = time.time()
    with torch.no_grad():
        out = m(x, t, encoder_hidden_states=text, encoder_attention_mask=mask, enable_temporal_attentions=temporal,
                return_dict=False)[0]
    res = dict(**G.pack("out", out.numpy()), t=t.numpy(), x_sum=np.float64(x.double().sum().item()),
               text_sum=np.float64(text.double().sum().item()),
               cfg=np.array(repr(cfg_kw)), batch=np.int64(batch), text_len=np.int64(text_len), wseed=np.int64(wseed),
               iseed=np.int64(iseed), temporal=np.int64(int(temporal)))
    if digest:
        res["weights_sha256"] = np.array(weights_digest(sd))
    if mask is not None:
        res["mask"] = mask.numpy()
    path = os.path.join(out_dir, f"t2v_{tag}.npz")
    np.savez_compressed(path, **res)
    print(f"{path}: out {tuple(out.shape)} absmax {out.abs().max():.4f} std {out.std():.4f}  ({time.time() - t0:.1f} s)")


def gen_subops(ref, out_dir):
    """Direct calls of the classes the reference file itself defines (plus the shim's spatial block for completeness)."""
    cfg = T.T2VConfig(num_attention_heads=4, attention_head_dim=72, num_layers=1, sample_size=16, video_length=8, caption_channels=256)
    sd = T.make_weights(cfg, 41)
    m = build_ref_model(ref, cfg, sd)
    D = cfg.inner_dim
    g = torch.Generator().manual_seed(77)
    xs = torch.randn(6, 8, D, generator=g)              # (B*N, F, D) rows for the temporal block
    ts = torch.randn(6, 6 * D, generator=g) * 0.3
    xsp = torch.randn(3, 64, D, generator=g)            # (B*F, N, D) rows for the spatial block
    tsp = torch.randn(3, 6 * D, generator=g) * 0.3
    txt = torch.randn(3, 20, D, generator=g)
    bias = torch.zeros(3, 1, 20)
    bias[1, 0, 7:] = -10000.0
    tt = torch.tensor([0, 17, 999])
    with torch.no_grad():
        ada, emb = m.adaln_single(tt, None, batch_size=3, hidden_dtype=torch.float32)
        res = dict(
            xs=xs.numpy(), ts=ts.numpy(), xsp=xsp.numpy(), tsp=tsp.numpy(), txt=txt.numpy(), bias=bias.numpy(), t=tt.numpy(),
            temporal_block0=m.temporal_transformer_blocks[0](xs, None, None, None, ts, None, None).numpy(),
            ff_temporal0=m.temporal_transformer_blocks[0].ff(xs).numpy(),
            adaln_single=ada.numpy(), embedded_timestep=emb.numpy(),
            temp_pos_embed=m.temp_pos_embed.numpy(),
            spatial_block0_shim=m.transformer_blocks[0](xsp, None, txt, None, tsp, None, None).numpy(),
            spatial_block0_masked_shim=m.transformer_blocks[0](xsp, None, txt, bias, tsp, None, None).numpy(),
            pos_embed_shim=m.pos_embed.pos_embed.numpy(),
        )
    np.savez_compressed(os.path.join(out_dir, "t2v_subops.npz"), **res)
    print("t2v_subops.npz written")


TINY = dict(num_attention_heads=2, attention_head_dim=64, num_layers=2, sample_size=16, video_length=8, caption_channels=256)
HD72 = dict(num_attention_heads=8, attention_head_dim=72, num_layers=2, sample_size=32, video_length=16, caption_channels=512)
S64 = dict(num_attention_heads=8, attention_head_dim=72, num_layers=2, sample_size=64, video_length=16, caption_channels=256)
FULL = dict(num_attention_heads=16, attention_head_dim=72, num_layers=28, sample_size=64, video_length=16, caption_channels=4096)

if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--full", action="store_true", help="also the Latte-1 shape: 28 layers, 16x512x512, L=120, batch 1")
    args = ap.parse_args()
    torch.manual_seed(0)
    out_dir = os.path.join(ROOT, "tests", "golden")
    ref = load_reference()
    gen_subops(ref, out_dir)
    gen_forward(ref, "tiny_b2_l20", TINY, 2, 20, 3, 4, out_dir)
    gen_forward(ref, "tiny_b2_l20_notemporal", TINY, 2, 20, 3, 4, out_dir, temporal=False)
    gen_forward(ref, "tiny_b2_l20_masked", TINY, 2, 20, 3, 4, out_dir, valid=[5, 20])
    gen_forward(ref, "hd72_b2_l120", HD72, 2, 120, 5, 6, out_dir)
    gen_forward(ref, "hd72_b2_l120_masked", HD72, 2, 120, 5, 6, out_dir, valid=[12, 120])
    gen_forward(ref, "s64_b1_l12", S64, 1, 12, 7, 8, out_dir)
    gen_forward(ref, "s64_b1_l120", S64, 1, 120, 7, 8, out_dir)
    if args.full:
        gen_forward(ref, "latte1_b1_l120", FULL, 1, 120, 0, 123, out_dir, digest=False)

"""CPU: the LatteT2V restatement (oracle/t2v_oracle.py) against goldens produced by the UNMODIFIED reference module
/root/reference/models/latte_t2v.py (oracle/make_golden_t2v.py, run through oracle/ref_shim/diffusers).  This pins the
forward control flow, the temporal block, adaLN-single, the feed-forward and the mask -> bias conversion to reference
code; the spatial block / Attention / PatchEmbed / CaptionProjection leaves are the shim's restatement of diffusers
0.24.0 (see the shim header).  Tolerance: same fp32 math in a different op order -> 5e-4 on O(5) outputs."""
import ast
import hashlib
import os

import numpy as np
import pytest
import torch

from oracle import golden as G
from oracle import t2v_oracle as T


def _digest(sd):
    h = hashlib.sha256()
    for k in sorted(sd):
        h.update(k.encode())
        h.update(sd[k].numpy().tobytes())
    return h.hexdigest()


def load_case(golden_dir, tag):
    g = np.load(os.path.join(golden_dir, f"t2v_{tag}.npz"))
    cfg = T.T2VConfig(**ast.literal_eval(str(g["cfg"])))
    sd = T.make_weights(cfg, int(g["wseed"]))
    if "weights_sha256" in g:
        assert _digest(sd) == str(g["weights_sha256"]), "seeded weights differ from the ones the golden was made with"
    x, t, text = T.make_inputs(cfg, int(g["batch"]), int(g["text_len"]), int(g["iseed"]))
    assert abs(float(x.double().sum()) - float(g["x_sum"])) < 1e-9 and abs(float(text.double().sum()) - float(g["text_sum"])) < 1e-9
    mask = torch.from_numpy(g["mask"]) if "mask" in g else None
    return g, cfg, sd, x, t, text, mask


CASES = ["tiny_b2_l20", "tiny_b2_l20_notemporal", "tiny_b2_l20_masked", "hd72_b2_l120", "hd72_b2_l120_masked", "s64_b1_l12",
         "s64_b1_l120"]


@pytest.mark.parametrize("tag", CASES)
def test_forward_matches_reference_golden(golden_dir, tag):
    g, cfg, sd, x, t, text, mask = load_case(golden_dir, tag)
    out = T.t2v_forward(sd, cfg, x, t, text, enable_temporal=bool(int(g["temporal"])), text_mask=mask)
    out, ref = G.pair(g, "out", out)
    assert (out - ref).abs().max().item() < 5e-4


def test_mask_changes_the_output(golden_dir):
    """the masked goldens are not the unmasked ones (the reference really applied the bias)"""
    shape, idx, a = G.stored(np.load(os.path.join(golden_dir, "t2v_hd72_b2_l120.npz")), "out")
    shape_m, idx_m, b = G.stored(np.load(os.path.join(golden_dir, "t2v_hd72_b2_l120_masked.npz")), "out")
    assert shape == shape_m and shape[0] == 2 and np.array_equal(idx, idx_m)
    d = np.abs(a - b)
    first = idx < np.prod(shape[1:])      # stored elements of sample 0
    assert d[first].max() > 1e-2          # sample 0 keeps 12 of 120 tokens
    assert d[~first].max() < 1e-5         # sample 1 keeps all of them


def test_subops_match_reference_classes(golden_dir):
    """BasicTransformerBlock_, FeedForward, AdaLayerNormSingle called directly on the reference's own classes."""
    g = np.load(os.path.join(golden_dir, "t2v_subops.npz"))
    cfg = T.T2VConfig(num_attention_heads=4, attention_head_dim=72, num_layers=1, sample_size=16, video_length=8, caption_channels=256)
    sd = T.make_weights(cfg, 41)
    xs, ts = torch.from_numpy(g["xs"]), torch.from_numpy(g["ts"])
    out = T.temporal_block(sd, 0, xs, ts, cfg.num_attention_heads)
    assert (out - torch.from_numpy(g["temporal_block0"])).abs().max().item() < 2e-4
    ff = T.feed_forward(sd, "temporal_transformer_blocks.0.ff", xs)
    assert (ff - torch.from_numpy(g["ff_temporal0"])).abs().max().item() < 2e-4
    ada, emb = T.adaln_single(sd, torch.from_numpy(g["t"]))
    assert (emb - torch.from_numpy(g["embedded_timestep"])).abs().max().item() < 2e-4
    assert (ada - torch.from_numpy(g["adaln_single"])).abs().max().item() < 2e-4
    assert np.abs(T.temp_pos_embed_table(cfg).numpy() - g["temp_pos_embed"][0]).max() < 1e-6
    # shim-restated leaves (diffusers): agreement here only says the two restatements agree
    xsp, tsp, txt = torch.from_numpy(g["xsp"]), torch.from_numpy(g["tsp"]), torch.from_numpy(g["txt"])
    sp = T.spatial_block(sd, 0, xsp, txt, tsp, cfg.num_attention_heads)
    assert (sp - torch.from_numpy(g["spatial_block0_shim"])).abs().max().item() < 2e-4
    spm = T.spatial_block(sd, 0, xsp, txt, tsp, cfg.num_attention_heads, torch.from_numpy(g["bias"])[:, 0])
    assert (spm - torch.from_numpy(g["spatial_block0_masked_shim"])).abs().max().item() < 2e-4
    assert np.abs(T.pos_embed_table(cfg).numpy() - g["pos_embed_shim"][0]).max() < 1e-6

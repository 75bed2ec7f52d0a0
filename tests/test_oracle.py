"""CPU: the oracle restatement (oracle/latte_oracle.py) against goldens produced by the UNMODIFIED
reference (oracle/make_golden.py).  This is the pin that lets the GPU parity tests trust the oracle."""
import hashlib
import os
import re

import numpy as np
import pytest
import torch

from oracle import golden as G
from oracle import latte_oracle as O


def _load(golden_dir, fname):
    g = np.load(os.path.join(golden_dir, fname))
    meta = str(g["meta"])
    m = re.match(r"(\S+) batch=(\d+) wseed=(\d+) iseed=(\d+) extras=(\d+) frames=(\d+) input=(\d+)", meta)
    name, batch, wseed, iseed, extras, frames, inp = m.group(1), *map(int, m.groups()[1:])
    cfg = O.make_config(name, extras=extras, num_frames=frames, input_size=inp)
    return g, cfg, batch, wseed, iseed


def _digest(sd):
    h = hashlib.sha256()
    for k in sorted(sd):
        h.update(k.encode())
        h.update(sd[k].numpy().tobytes())
    return h.hexdigest()


FWD = ["latte_tiny64_2_b2.npz", "latte_tiny72_2_b2.npz", "latte_tiny72_2_extras1_b4.npz", "latte_s_2_b2.npz"]


@pytest.mark.parametrize("fname", FWD)
def test_forward_matches_reference_golden(golden_dir, fname):
    g, cfg, batch, wseed, iseed = _load(golden_dir, fname)
    sd = O.make_weights(cfg, wseed)
    assert _digest(sd) == str(g["weights_sha256"]), "seeded weights differ from the ones the golden was made with"
    x, t, y = O.make_inputs(cfg, batch, iseed)
    assert abs(float(x.double().sum()) - float(g["x_sum"])) < 1e-9
    out = O.latte_forward(sd, cfg, x, t, y)
    assert out.shape == (batch, cfg.num_frames, cfg.out_channels, cfg.input_size, cfg.input_size)
    got, ref = G.pair(g, "out", out)
    # same fp32 math, different op order (fused reshape vs einops): tolerance 2e-4 on O(5) outputs
    assert (got - ref).abs().max().item() < 2e-4
    out_cfg = O.latte_forward_with_cfg(sd, cfg, x, t, y, cfg_scale=7.0)
    half = torch.from_numpy(g["out_cfg_half_eps"])
    assert (out_cfg[: batch // 2, :, :4] - half).abs().max().item() < 1e-3
    # both halves carry the same guided eps; 'rest' channels are the raw model output (latte.py:394-398)
    assert torch.equal(out_cfg[: batch // 2, :, :4], out_cfg[batch // 2:, :, :4])


def test_fp64_oracle_is_closer_than_bf16_reference(golden_dir):
    """The reference's own bf16-autocast deviation is the noise floor the GPU tolerance is judged against."""
    g, cfg, batch, wseed, iseed = _load(golden_dir, "latte_tiny72_2_b2.npz")
    sd = O.make_weights(cfg, wseed)
    x, t, y = O.make_inputs(cfg, batch, iseed)
    got, ref = G.pair(g, "out", O.latte_forward(sd, cfg, x.double(), t, y, dtype=torch.float64).float())
    dev = (got - ref).abs().max().item()
    assert dev < 2e-4 < float(g["ref_bf16_maxabs"])


def test_subops_match_reference(golden_dir):
    g = np.load(os.path.join(golden_dir, "subops_tiny72.npz"))
    cfg = O.make_config("Latte-tiny72/2", input_size=16, num_frames=4)
    sd = O.make_weights(cfg, 7)
    xs, c = O.subops_inputs(cfg)
    assert abs(float(xs.double().sum()) - float(g["xs_sum"])) < 1e-9
    assert torch.equal(c, torch.from_numpy(g["c"]))
    t = torch.from_numpy(g["t"])
    tol = 2e-5

    def err(key, got):
        got, want = G.pair(g, key, got)
        return (got - want).abs().max()
    assert (O.timestep_embedding(t) - torch.from_numpy(g["t_freq"])).abs().max() < 1e-6
    assert (O.t_embedder(sd, t, torch.float32) - torch.from_numpy(g["t_emb"])).abs().max() < tol
    assert err("block0", O.transformer_block(sd, 0, xs, c, cfg.num_heads)) < 1e-4
    assert err("attn0", O.attention_math(sd, "blocks.0.attn.", xs, cfg.num_heads)) < tol
    assert err("mlp0", O.mlp(sd, "blocks.0.mlp.", xs)) < tol
    assert (O.final_layer(sd, xs, c) - torch.from_numpy(g["final"])).abs().max() < 1e-4
    assert err("modulate", O.modulate(O.layer_norm(xs), c, c * 0.5)) < tol
    un = O.unpatchify(cfg, torch.arange(2 * 64 * 32, dtype=torch.float32).reshape(2, 64, 32))
    assert torch.equal(un, torch.from_numpy(g["unpatchify"]))
    # sin-cos tables: bit-exact against a freshly initialised reference model
    assert np.array_equal(sd["pos_embed"].numpy(), g["fresh_pos_embed"])
    assert np.array_equal(sd["temp_embed"].numpy(), g["fresh_temp_embed"])
    # F5: the reference's own init gives an all-zero output, which is why make_weights is not that init
    assert float(g["fresh_out_absmax"]) == 0.0


def test_state_dict_contract():
    """SURVEY.md App. B: 13 + 10*depth tensors with extras==2, 12 + 10*depth without."""
    cfg = O.make_config("Latte-S/2")
    assert len(O.state_dict_spec(cfg)) == 13 + 10 * cfg.depth == 133
    cfg1 = O.make_config("Latte-S/2", extras=1)
    assert len(O.state_dict_spec(cfg1)) == 12 + 10 * cfg1.depth


def test_algorithmic_flops_match_survey():
    """SURVEY.md App. A: S/2 0.1844 TFLOP, XL/2 3.7256 TFLOP per video per forward."""
    assert abs(O.algorithmic_flops_per_video(O.make_config("Latte-S/2")) / 1e12 - 0.1844) < 2e-4
    assert abs(O.algorithmic_flops_per_video(O.make_config("Latte-XL/2")) / 1e12 - 3.7256) < 2e-4

"""CPU oracle for the Latte denoiser forward — TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Only `tests/`, `__graft_entry__.smoke()` and `bench.py`'s cpu_baseline / `--impl reference`
legs may import this file.  The product path (`latte_b200/`) never does and has no CPU fallback.

It is a functional restatement (plain torch CPU tensor ops, fp32 or fp64) of the algorithm in
`/root/reference/models/latte.py` (Vchitect/Latte @ b27c24a).  Every function cites the
reference lines it follows.  Parity status: the reference ships no tests / golden vectors
(SURVEY.md §4), so the pin is reference-generated: `oracle/make_golden.py` runs the UNMODIFIED
reference module (imported from /root/reference with the timm shim in `oracle/ref_shim`) on
the seeded weights/inputs defined here and commits its outputs under `tests/golden/`;
`tests/test_oracle.py` checks this restatement against those files on every run.

Third-party pieces restated here (not vendored in the reference): timm `Mlp` / `PatchEmbed`
(unpinned in environment.yml:12; semantics in SURVEY.md App. C.1).
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import numpy as np
import torch
import torch.nn.functional as F


# ----------------------------------------------------------------------------------------------
# configuration  (reference: models/latte.py:464-506 size table, :208-223 ctor signature)
# ----------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class LatteConfig:
    input_size: int = 32
    patch_size: int = 2
    in_channels: int = 4
    hidden_size: int = 1152
    depth: int = 28
    num_heads: int = 16
    mlp_ratio: float = 4.0
    num_frames: int = 16
    num_classes: int = 101
    learn_sigma: bool = True
    extras: int = 2
    class_dropout_prob: float = 0.1

    @property
    def out_channels(self) -> int:  # latte.py:227
        return self.in_channels * 2 if self.learn_sigma else self.in_channels

    @property
    def num_patches(self) -> int:
        return (self.input_size // self.patch_size) ** 2

    @property
    def head_dim(self) -> int:
        return self.hidden_size // self.num_heads


CONFIGS = {
    # latte.py:464-465 / :497-498 (depth, hidden, heads) — patch 2 variants only
    "Latte-XL/2": dict(depth=28, hidden_size=1152, num_heads=16),
    "Latte-L/2": dict(depth=24, hidden_size=1024, num_heads=16),
    "Latte-B/2": dict(depth=12, hidden_size=768, num_heads=12),
    "Latte-S/2": dict(depth=12, hidden_size=384, num_heads=6),
    # not in the reference table: a 4-block model with XL's awkward head_dim (72) for fast tests
    "Latte-tiny72/2": dict(depth=4, hidden_size=576, num_heads=8),
    "Latte-tiny64/2": dict(depth=2, hidden_size=128, num_heads=2),
}


def make_config(name: str, **kw) -> LatteConfig:
    return LatteConfig(**CONFIGS[name], **kw)


# ----------------------------------------------------------------------------------------------
# sin-cos tables (latte.py:406-457) — numpy fp64 → fp32, exactly as the reference builds them
# ----------------------------------------------------------------------------------------------
def sincos_1d_from_grid(embed_dim: int, pos: np.ndarray) -> np.ndarray:  # latte.py:440-457
    omega = np.arange(embed_dim // 2, dtype=np.float64)
    omega /= embed_dim / 2.0
    omega = 1.0 / 10000 ** omega
    out = np.einsum("m,d->md", pos.reshape(-1), omega)
    return np.concatenate([np.sin(out), np.cos(out)], axis=1)


def sincos_2d(embed_dim: int, grid_size: int) -> np.ndarray:  # latte.py:410-438
    grid_h = np.arange(grid_size, dtype=np.float32)
    grid_w = np.arange(grid_size, dtype=np.float32)
    grid = np.stack(np.meshgrid(grid_w, grid_h), axis=0).reshape([2, 1, grid_size, grid_size])
    emb_h = sincos_1d_from_grid(embed_dim // 2, grid[0])
    emb_w = sincos_1d_from_grid(embed_dim // 2, grid[1])
    return np.concatenate([emb_h, emb_w], axis=1)


def sincos_temp(embed_dim: int, length: int) -> np.ndarray:  # latte.py:406-408
    pos = np.arange(0, length, dtype=np.int64).reshape(-1, 1)
    return sincos_1d_from_grid(embed_dim, pos)


# ----------------------------------------------------------------------------------------------
# deterministic weights with the reference's state_dict key names (SURVEY.md App. B)
# ----------------------------------------------------------------------------------------------
def state_dict_spec(cfg: LatteConfig):
    """(name, shape) in a fixed order — the reference's key set (latte.py:233-255)."""
    D, p, C = cfg.hidden_size, cfg.patch_size, cfg.in_channels
    H4 = int(D * cfg.mlp_ratio)
    spec = [
        ("pos_embed", (1, cfg.num_patches, D)),
        ("temp_embed", (1, cfg.num_frames, D)),
        ("x_embedder.proj.weight", (D, C, p, p)),
        ("x_embedder.proj.bias", (D,)),
        ("t_embedder.mlp.0.weight", (D, 256)),
        ("t_embedder.mlp.0.bias", (D,)),
        ("t_embedder.mlp.2.weight", (D, D)),
        ("t_embedder.mlp.2.bias", (D,)),
    ]
    if cfg.extras == 2:
        spec.append(("y_embedder.embedding_table.weight",
                     (cfg.num_classes + (1 if cfg.class_dropout_prob > 0 else 0), D)))
    for i in range(cfg.depth):
        b = f"blocks.{i}."
        spec += [
            (b + "attn.qkv.weight", (3 * D, D)), (b + "attn.qkv.bias", (3 * D,)),
            (b + "attn.proj.weight", (D, D)), (b + "attn.proj.bias", (D,)),
            (b + "mlp.fc1.weight", (H4, D)), (b + "mlp.fc1.bias", (H4,)),
            (b + "mlp.fc2.weight", (D, H4)), (b + "mlp.fc2.bias", (D,)),
            (b + "adaLN_modulation.1.weight", (6 * D, D)), (b + "adaLN_modulation.1.bias", (6 * D,)),
        ]
    spec += [
        ("final_layer.linear.weight", (p * p * cfg.out_channels, D)),
        ("final_layer.linear.bias", (p * p * cfg.out_channels,)),
        ("final_layer.adaLN_modulation.1.weight", (2 * D, D)),
        ("final_layer.adaLN_modulation.1.bias", (2 * D,)),
    ]
    return spec


def make_weights(cfg: LatteConfig, seed: int = 0) -> dict[str, torch.Tensor]:
    """Seeded fp32 weights.  NOT the reference initialiser: `initialize_weights`
    (latte.py:286-295) zeroes every adaLN / final linear, so a fresh model outputs exactly 0
    (SURVEY.md F5) and parity would compare 0 with 0.  Instead every matrix gets
    N(0, 1/fan_in) scaled per family so all paths carry signal at O(1) magnitudes, and every bias is
    non-zero.  pos/temp embeds are the reference's sin-cos tables."""
    g = torch.Generator().manual_seed(seed)
    D = cfg.hidden_size
    sd = {}
    for name, shape in state_dict_spec(cfg):
        if name == "pos_embed":
            t = torch.from_numpy(sincos_2d(D, int(cfg.num_patches ** 0.5))).float().unsqueeze(0)
        elif name == "temp_embed":
            t = torch.from_numpy(sincos_temp(D, cfg.num_frames)).float().unsqueeze(0)
        elif name.endswith(".bias"):
            t = torch.randn(shape, generator=g) * 0.05
        elif name == "y_embedder.embedding_table.weight":
            t = torch.randn(shape, generator=g) * 0.5
        elif name == "x_embedder.proj.weight":
            t = torch.randn(shape, generator=g) * 0.25
        elif "adaLN_modulation" in name:
            t = torch.randn(shape, generator=g) * (0.5 / math.sqrt(shape[1]))
        else:
            t = torch.randn(shape, generator=g) * (1.0 / math.sqrt(shape[-1]))
        sd[name] = t.contiguous()
    return sd


def make_inputs(cfg: LatteConfig, batch: int, seed: int = 123):
    """Seeded (x, t, y).  Last row gets the null class (sample.py:90-92 puts it in the 2nd half)."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(batch, cfg.num_frames, cfg.in_channels, cfg.input_size, cfg.input_size, generator=g)
    t = torch.randint(0, 1000, (batch,), generator=g)
    y = torch.randint(0, cfg.num_classes, (batch,), generator=g)
    y[batch // 2:] = cfg.num_classes
    return x, t, y


def subops_inputs(cfg: LatteConfig, seed: int = 99):
    """Seeded (xs, c) of the sub-op goldens: 3 sequences of 64 tokens and their conditioning vectors."""
    g = torch.Generator().manual_seed(seed)
    xs = torch.randn(3, 64, cfg.hidden_size, generator=g)
    c = torch.randn(3, cfg.hidden_size, generator=g)
    return xs, c


# ----------------------------------------------------------------------------------------------
# the forward, op by op
# ----------------------------------------------------------------------------------------------
def timestep_embedding(t: torch.Tensor, dim: int = 256, max_period: int = 10000) -> torch.Tensor:
    """latte.py:98-116 — [cos(t w_k), sin(t w_k)], w_k = exp(-ln(1e4) k / half); fp32 like the reference."""
    half = dim // 2
    freqs = torch.exp(-math.log(max_period) * torch.arange(0, half, dtype=torch.float32) / half).to(device=t.device)
    args = t[:, None].float() * freqs[None]
    return torch.cat([torch.cos(args), torch.sin(args)], dim=-1)


def t_embedder(sd, t, dtype):
    """latte.py:118-123 — Linear(256,D) → SiLU → Linear(D,D)."""
    h = timestep_embedding(t).to(dtype)
    h = F.linear(h, sd["t_embedder.mlp.0.weight"].to(dtype), sd["t_embedder.mlp.0.bias"].to(dtype))
    h = F.silu(h)
    return F.linear(h, sd["t_embedder.mlp.2.weight"].to(dtype), sd["t_embedder.mlp.2.bias"].to(dtype))


def y_embedder(sd, y, dtype):
    """latte.py:148-153 in eval mode (no token drop): a table lookup."""
    return sd["y_embedder.embedding_table.weight"].to(dtype)[y]


def patch_embed(sd, cfg, x, dtype):
    """latte.py:330-331 + timm PatchEmbed: Conv2d(k=s=p) == per-patch GEMM (K = C p p), then + pos_embed."""
    B, Fr, C, Hh, Ww = x.shape
    p = cfg.patch_size
    xx = x.reshape(B * Fr, C, Hh // p, p, Ww // p, p).permute(0, 2, 4, 1, 3, 5)  # n, gh, gw, c, i, j
    xx = xx.reshape(B * Fr, (Hh // p) * (Ww // p), C * p * p).to(dtype)
    w = sd["x_embedder.proj.weight"].to(dtype).reshape(cfg.hidden_size, C * p * p)
    tok = xx @ w.t() + sd["x_embedder.proj.bias"].to(dtype)
    return tok + sd["pos_embed"].to(dtype)


def layer_norm(x, eps=1e-6):
    """latte.py:166,168,189 — LayerNorm(elementwise_affine=False, eps=1e-6): biased variance."""
    mu = x.mean(dim=-1, keepdim=True)
    var = ((x - mu) ** 2).mean(dim=-1, keepdim=True)
    return (x - mu) / torch.sqrt(var + eps)


def modulate(x, shift, scale):
    """latte.py:28-29."""
    return x * (1 + scale.unsqueeze(1)) + shift.unsqueeze(1)


def attention_math(sd, prefix, x, num_heads):
    """latte.py:48-77, attention_mode='math' (the only mode any script reaches — SURVEY.md F4)."""
    Bs, S, C = x.shape
    hd = C // num_heads
    dtype = x.dtype
    qkv = F.linear(x, sd[prefix + "qkv.weight"].to(dtype), sd[prefix + "qkv.bias"].to(dtype))
    qkv = qkv.reshape(Bs, S, 3, num_heads, hd).permute(2, 0, 3, 1, 4)
    q, k, v = qkv[0], qkv[1], qkv[2]
    attn = (q @ k.transpose(-2, -1)) * (hd ** -0.5)
    attn = attn.softmax(dim=-1)
    o = (attn @ v).transpose(1, 2).reshape(Bs, S, C)
    return F.linear(o, sd[prefix + "proj.weight"].to(dtype), sd[prefix + "proj.bias"].to(dtype))


def mlp(sd, prefix, x):
    """latte.py:169-171 + timm Mlp: fc1 → GELU(approximate='tanh') → fc2."""
    dtype = x.dtype
    h = F.linear(x, sd[prefix + "fc1.weight"].to(dtype), sd[prefix + "fc1.bias"].to(dtype))
    h = F.gelu(h, approximate="tanh")
    return F.linear(h, sd[prefix + "fc2.weight"].to(dtype), sd[prefix + "fc2.bias"].to(dtype))


def transformer_block(sd, i, x, c, num_heads):
    """latte.py:177-181 — adaLN-Zero block.  x: (Bs,S,D), c: (Bs,D)."""
    p = f"blocks.{i}."
    dtype = x.dtype
    mod = F.linear(F.silu(c), sd[p + "adaLN_modulation.1.weight"].to(dtype),
                   sd[p + "adaLN_modulation.1.bias"].to(dtype))
    shift_msa, scale_msa, gate_msa, shift_mlp, scale_mlp, gate_mlp = mod.chunk(6, dim=1)
    x = x + gate_msa.unsqueeze(1) * attention_math(sd, p + "attn.", modulate(layer_norm(x), shift_msa, scale_msa), num_heads)
    x = x + gate_mlp.unsqueeze(1) * mlp(sd, p + "mlp.", modulate(layer_norm(x), shift_mlp, scale_mlp))
    return x


def final_layer(sd, x, c):
    """latte.py:197-201."""
    dtype = x.dtype
    mod = F.linear(F.silu(c), sd["final_layer.adaLN_modulation.1.weight"].to(dtype),
                   sd["final_layer.adaLN_modulation.1.bias"].to(dtype))
    shift, scale = mod.chunk(2, dim=1)
    x = modulate(layer_norm(x), shift, scale)
    return F.linear(x, sd["final_layer.linear.weight"].to(dtype), sd["final_layer.linear.bias"].to(dtype))


def unpatchify(cfg, x):
    """latte.py:297-310 — (n, T, p*p*c) → (n, c, h*p, w*p); channel is the fastest of (p, q, c)."""
    c, p = cfg.out_channels, cfg.patch_size
    h = w = int(x.shape[1] ** 0.5)
    x = x.reshape(x.shape[0], h, w, p, p, c)
    x = torch.einsum("nhwpqc->nchpwq", x)
    return x.reshape(x.shape[0], c, h * p, w * p)


def latte_forward(sd, cfg: LatteConfig, x, t, y=None, dtype=torch.float32, return_hidden=False):
    """latte.py:314-377 (eval mode, extras in {1, 2})."""
    B, Fr = x.shape[0], x.shape[1]
    N, D = cfg.num_patches, cfg.hidden_size
    h = patch_embed(sd, cfg, x, dtype)                       # (B*F, N, D)   :330-331
    c = t_embedder(sd, t, dtype)                             # (B, D)        :332
    if cfg.extras == 2:
        c = c + y_embedder(sd, y, dtype)                     # :337, :348
    c_spatial = c.repeat_interleave(Fr, dim=0)               # :333,:338  'n d -> (n c) d'
    c_temp = c.repeat_interleave(N, dim=0)                   # :334,:339
    for i in range(0, cfg.depth, 2):                         # :345
        h = transformer_block(sd, i, h, c_spatial, cfg.num_heads)                     # :353
        h = h.reshape(B, Fr, N, D).permute(0, 2, 1, 3).reshape(B * N, Fr, D)          # :355
        if i == 0:
            h = h + sd["temp_embed"].to(dtype)                                        # :357-358
        h = transformer_block(sd, i + 1, h, c_temp, cfg.num_heads)                    # :367
        h = h.reshape(B, N, Fr, D).permute(0, 2, 1, 3).reshape(B * Fr, N, D)          # :368
    hidden = h
    o = final_layer(sd, h, c_spatial)                        # :374
    o = unpatchify(cfg, o)                                   # :375
    o = o.reshape(B, Fr, *o.shape[1:])                       # :376
    return (o, hidden) if return_hidden else o


def latte_forward_with_cfg(sd, cfg: LatteConfig, x, t, y=None, cfg_scale=7.0, dtype=torch.float32):
    """latte.py:379-398 — guidance on channels [:4] only; both halves get the guided eps."""
    half = x[: len(x) // 2]
    combined = torch.cat([half, half], dim=0)
    out = latte_forward(sd, cfg, combined, t, y, dtype)
    eps, rest = out[:, :, :4], out[:, :, 4:]
    cond, uncond = torch.split(eps, len(eps) // 2, dim=0)
    half_eps = uncond + cfg_scale * (cond - uncond)
    return torch.cat([torch.cat([half_eps, half_eps], dim=0), rest], dim=2)


# ----------------------------------------------------------------------------------------------
# algorithmic FLOPs (SURVEY.md App. A) — used by bench.py for the roofline numerator
# ----------------------------------------------------------------------------------------------
def algorithmic_flops_per_video(cfg: LatteConfig) -> float:
    D, N, Fr, L = cfg.hidden_size, cfg.num_patches, cfg.num_frames, cfg.depth
    T = N * Fr
    H4 = int(D * cfg.mlp_ratio)
    lin = 2.0 * T * (D * 3 * D + D * D + 2 * D * H4) * L
    attn = (4.0 * N * N * D * Fr + 4.0 * Fr * Fr * D * N) * (L // 2)
    ada = 2.0 * D * 6 * D * L + 2.0 * D * 2 * D
    emb = 2.0 * T * (cfg.in_channels * cfg.patch_size ** 2) * D + 2.0 * T * D * (cfg.patch_size ** 2 * cfg.out_channels)
    return lin + attn + ada + emb

"""GPU parity of the whole denoiser forward through the C ABI against (1) goldens produced by the unmodified
reference and (2) the CPU oracle, plus size-independent properties at the BASELINE shape.

Tolerance (stated per north_star): max-abs < 1e-2 on outputs of magnitude ~5 for fp16 operands
(measured 1.5e-3 on XL/2); bf16 operands are held to the reference's OWN bf16-autocast deviation on the same
weights (stored in the golden as ref_bf16_maxabs, 2-3e-2) — bf16 cannot meet 1e-2 in the reference either."""
import os
import re

import numpy as np
import pytest
import torch

from oracle import golden as G
from oracle import latte_oracle as O

pytestmark = pytest.mark.gpu


def _build(golden_dir, fname):
    from latte_b200 import Latte
    from oracle import latte_oracle as O
    g = np.load(os.path.join(golden_dir, fname))
    m = re.match(r"(\S+) batch=(\d+) wseed=(\d+) iseed=(\d+) extras=(\d+) frames=(\d+) input=(\d+)", str(g["meta"]))
    name, batch, wseed, iseed, extras, frames, inp = m.group(1), *map(int, m.groups()[1:])
    cfg = O.make_config(name, extras=extras, num_frames=frames, input_size=inp)
    sd = O.make_weights(cfg, wseed)
    x, t, y = O.make_inputs(cfg, batch, iseed)
    net = Latte(input_size=cfg.input_size, hidden_size=cfg.hidden_size, depth=cfg.depth, num_heads=cfg.num_heads,
                num_frames=cfg.num_frames, num_classes=cfg.num_classes, learn_sigma=True, extras=cfg.extras)
    net.load_state_dict(sd, strict=True)
    return g, cfg, sd, net.to("cuda:0").eval(), (x, t, y if extras == 2 else None)


CASES = ["latte_tiny64_2_b2.npz", "latte_tiny72_2_b2.npz", "latte_tiny72_2_extras1_b4.npz", "latte_s_2_b2.npz", "latte_xl_2_b2.npz"]


@pytest.mark.parametrize("fname", CASES)
def test_forward_matches_reference_golden(golden_dir, fname):
    g, cfg, sd, net, (x, t, y) = _build(golden_dir, fname)
    half = torch.from_numpy(g["out_cfg_half_eps"])
    dev = torch.device("cuda:0")
    xd, td, yd = x.to(dev), t.to(dev), (y.to(dev) if y is not None else None)
    with torch.no_grad():
        for dt, tol in ((torch.float16, 1e-2), (torch.bfloat16, float(g["ref_bf16_maxabs"]))):
            net.compute_dtype = dt
            out = net(xd, td, y=yd).cpu()
            assert out.dtype == torch.float32
            got, ref = G.pair(g, "out", out)
            err = (got - ref).abs().max().item()
            assert err < tol, f"{fname} {dt}: max-abs {err:.3e} >= {tol:.3e}"
            oc = net.forward_with_cfg(xd, td, y=yd, cfg_scale=7.0).cpu()
            b = out.shape[0]
            # guidance amplifies the deviation by (2 * 7 - 1): eps = u + 7 (c - u)
            assert (oc[: b // 2, :, :4] - half).abs().max().item() < 13 * tol
            assert torch.equal(oc[: b // 2, :, :4], oc[b // 2:, :, :4])
    # the half model (module.half(), sample.py:72-75) returns fp16 like the reference
    net.half()
    with torch.no_grad():
        o16 = net(xd, td, y=yd)
    got, ref = G.pair(g, "out", o16.float().cpu())
    assert o16.dtype == torch.float16 and (got - ref).abs().max().item() < 1.5e-2   # vs the fp32-weight golden: includes the weight rounding
    if "xl" not in fname:
        # the north_star bound (1e-2) on the path itself: against the oracle evaluated in fp32 on the SAME fp16-rounded weights
        # (sample.py:72-75's model.half()), so that only the kernels' operand rounding is measured
        sd_h = {k: (v.half().float() if v.dtype == torch.float32 else v) for k, v in sd.items()}      # .half() rounds every parameter
        ref_h = O.latte_forward(sd_h, cfg, x, t, y)
        err_h = (o16.float().cpu() - ref_h).abs().max().item()
        assert err_h < 1e-2, f"{fname} .half(): max-abs {err_h:.3e} vs the fp32 oracle on fp16-rounded weights"


def test_forward_matches_cpu_oracle_fresh_seed(golden_dir):
    """Not a stored vector: new seeds through the oracle restatement (pinned to the reference by tests/test_oracle.py)."""
    from latte_b200 import Latte
    from oracle import latte_oracle as O
    cfg = O.make_config("Latte-tiny72/2", input_size=16, num_frames=16)
    sd = O.make_weights(cfg, 77)
    x, t, y = O.make_inputs(cfg, 3, 78)
    net = Latte(input_size=16, hidden_size=cfg.hidden_size, depth=cfg.depth, num_heads=cfg.num_heads, num_frames=16,
                num_classes=cfg.num_classes, extras=2)
    net.load_state_dict(sd)
    net = net.cuda().eval()
    with torch.no_grad():
        out = net(x.cuda(), t.cuda(), y=y.cuda()).cpu()
    assert (out - O.latte_forward(sd, cfg, x, t, y)).abs().max().item() < 1e-2


def test_properties_at_baseline_shape(golden_dir):
    """XL/2, 16x4x32x32 (BASELINE configs[1]): batch rows are independent, reruns are bit-identical, cfg_scale=1 returns
    the conditional eps, and the zero-initialised reference model returns exactly 0 (adaLN-Zero, SURVEY.md F5)."""
    from latte_b200 import Latte_models
    g, cfg, sd, net, (x, t, y) = _build(golden_dir, "latte_xl_2_b2.npz")
    dev = torch.device("cuda:0")
    xd, td, yd = x.to(dev), t.to(dev), y.to(dev)
    with torch.no_grad():
        full = net(xd, td, y=yd)
        assert torch.equal(full, net(xd, td, y=yd))
        solo = net(xd[1:], td[1:], y=yd[1:])
        # no cross-sample coupling (attention is per sample).  Not bit-equal: the residual GEMMs split K differently for
        # M = 4096 and M = 8192 rows (stream-K), and a 1-ulp change of the fp32 stream can flip 16-bit operand roundings
        # downstream, so the two runs differ by 16-bit rounding noise (same size as the error against the fp32 golden)
        assert (solo - full[1:]).abs().max().item() < 5e-3
        c1 = net.forward_with_cfg(xd, td, y=yd, cfg_scale=1.0)
        twice = net(torch.cat([xd[:1], xd[:1]]), td, y=yd)
        assert (c1[:1, :, :4] - twice[:1, :, :4]).abs().max().item() < 1e-4
        assert torch.equal(c1[:, :, 4:], twice[:, :, 4:])
        fresh = Latte_models["Latte-S/2"](input_size=32, num_classes=101, num_frames=16, learn_sigma=True, extras=2).to(dev).eval()
        z = fresh(xd, td, y=yd)
        assert float(z.abs().max()) == 0.0


def test_sampler_drives_the_module(golden_dir):
    """A few DDIM-style steps calling the module exactly as gaussian_diffusion.p_mean_variance does (:279):
    `model(x, t, **model_kwargs)` with fp32 x, int64 t on device, kwargs y / cfg_scale — output (B,F,2C,H,W) (:290)."""
    g, cfg, sd, net, (x, t, y) = _build(golden_dir, "latte_tiny72_2_b2.npz")
    dev = torch.device("cuda:0")
    xs = x.to(dev)
    kwargs = dict(y=y.to(dev), cfg_scale=7.0, use_fp16=False)
    with torch.no_grad():
        for ti in (999, 995, 991):
            tt = torch.tensor([ti] * xs.shape[0], device=dev)
            out = net.forward_with_cfg(xs, tt, **kwargs)
            B, C = xs.shape[0], xs.shape[2]
            assert out.shape == (B, cfg.num_frames, 2 * C, cfg.input_size, cfg.input_size)
            eps, _ = torch.split(out, C, dim=2)
            xs = xs - 0.01 * eps
    assert torch.isfinite(xs).all()

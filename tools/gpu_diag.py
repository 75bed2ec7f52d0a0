"""GPU bring-up diagnostics (run under gpurun): staged probes of each kernel through the C ABI with
error PATTERNS, not just pass/fail, so a wrong descriptor/swizzle can be diagnosed from one run.
Usage: python tools/gpu_diag.py <stage>   stages: ln gemm_probe gemm attn_probe attn model xl
"""
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from latte_b200 import ops  # noqa: E402

dev = torch.device("cuda:0")
OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out")
os.makedirs(OUT, exist_ok=True)


def stat(name, got, ref, tol):
    got, ref = got.float(), ref.float()
    err = (got - ref).abs()
    bad = (err > tol + tol * ref.abs())
    print(f"[{'OK ' if not bad.any() else 'BAD'}] {name}: maxabs {err.max().item():.4e} mean {err.mean().item():.3e} "
          f"ref absmax {ref.abs().max().item():.3f} bad {bad.float().mean().item() * 100:.2f}% nan {torch.isnan(got).sum().item()}",
          flush=True)
    return bad


def stage_ln():
    g = torch.Generator(device="cpu").manual_seed(1)
    for D in (128, 384, 576, 1152):
        rows, B = 96, 3
        x = (torch.randn(rows, D, generator=g) * 2 + 0.5).to(dev)
        mod = torch.randn(B, 6 * D, generator=g).to(dev)
        shift, scale = mod[:, :D], mod[:, D:2 * D]
        for dt in (torch.float16, torch.bfloat16):
            out = ops.ln_modulate(x, shift, scale, rows // B, dt)
            xn = torch.nn.functional.layer_norm(x, (D,), eps=1e-6)
            b = torch.arange(rows, device=dev) // (rows // B)
            ref = xn * (1 + scale[b]) + shift[b]
            stat(f"ln_modulate D={D} {dt}", out, ref, 2e-3 if dt == torch.float16 else 1.6e-2)


def stage_gemm_probe():
    """W = [I_64; 0] so out[:, n<64] must equal A[:, n]; any permutation shows up as a column map."""
    for dt in (torch.float16,):
        M, N, K = 128, 128, 64
        A = (torch.arange(M * K, dtype=torch.float32).reshape(M, K) % 251 - 125).to(dev).to(dt)
        W = torch.zeros(N, K, device=dev, dtype=dt)
        W[:K, :K] = torch.eye(K, device=dev, dtype=dt)
        out = ops.linear(A, W, None, block_n=128)
        torch.cuda.synchronize()
        ref = A.float() @ W.float().t()
        bad = stat("gemm probe identity 128x128x64", out, ref, 1e-3)
        if bad.any():
            o = out.float().cpu().numpy()
            a = A.float().cpu().numpy()
            np.save(os.path.join(OUT, "probe_out.npy"), o)
            # for a few rows, say which A column each output column equals
            for r in (0, 1, 7, 8, 9, 64, 127):
                m = []
                for n in range(0, 64, 8):
                    hits = np.where(np.abs(a[r] - o[r, n]) < 1e-3)[0]
                    m.append(int(hits[0]) if len(hits) else -1)
                print(f"   row {r}: out cols 0,8,..56 come from A cols {m}; out[r,:4]={o[r,:4]} a[r,:4]={a[r,:4]}")
            print("   rows all-zero:", int((np.abs(o).sum(1) == 0).sum()), " cols>=64 nonzero:", int((np.abs(o[:, 64:]) > 0).sum()))


def stage_gemm():
    g = torch.Generator(device="cpu").manual_seed(2)
    cases = [(128, 128, 64), (128, 256, 128), (256, 384, 1152), (200, 192, 192), (1024, 1152, 1152), (640, 4608, 1152), (512, 1152, 4608)]
    for (M, N, K) in cases:
        for dt in (torch.float16, torch.bfloat16):
            A = torch.randn(M, K, generator=g).to(dev).to(dt)
            W = (torch.randn(N, K, generator=g) / K ** 0.5).to(dev).to(dt)
            bias = torch.randn(N, generator=g).to(dev)
            ref = A.float() @ W.float().t() + bias
            tol = 4e-3 if dt == torch.float16 else 3e-2
            for bn in (128, 192, 256):
                out = ops.linear(A, W, bias, block_n=bn)
                stat(f"gemm {M}x{N}x{K} {str(dt)[6:]} bn{bn}", out, ref, tol)
            out = ops.linear(A, W, bias, gelu=True)
            stat(f"gemm+gelu {M}x{N}x{K} {str(dt)[6:]} auto", out, torch.nn.functional.gelu(ref, approximate='tanh'), tol)
            B = 2
            rpb = (M + B - 1) // B
            gate = torch.randn(B, N, generator=g).to(dev)
            resid = torch.randn(M, N, generator=g).to(dev)
            want = resid + gate[torch.arange(M, device=dev) // rpb] * ref
            ops.linear_gate_residual_(resid, A, W, bias, gate, rpb)
            stat(f"gemm+gate_resid {M}x{N}x{K} {str(dt)[6:]} auto", resid, want, 5e-3 if dt == torch.float16 else 3e-2)


def attn_ref(qkv, batch, frames, tokens, heads, temporal):
    T, D3 = qkv.shape
    D = D3 // 3
    hd = D // heads
    x = qkv.float().reshape(batch, frames, tokens, 3, heads, hd)
    if temporal:
        x = x.permute(3, 0, 2, 4, 1, 5)   # 3, b, n, h, f, hd
    else:
        x = x.permute(3, 0, 1, 4, 2, 5)   # 3, b, f, h, n, hd
    q, k, v = x[0], x[1], x[2]
    a = torch.softmax(q @ k.transpose(-1, -2) * hd ** -0.5, dim=-1)
    o = a @ v                              # b, (n|f), h, (f|n), hd
    if temporal:
        o = o.permute(0, 3, 1, 2, 4)       # b, f, n, h, hd
    else:
        o = o.permute(0, 1, 3, 2, 4)       # b, f, n, h, hd
    return o.reshape(T, D)


def stage_attn_probe():
    g = torch.Generator(device="cpu").manual_seed(3)
    dt = torch.float16
    for (b, f, n, h, hd, temporal, label) in [(1, 1, 128, 1, 64, False, "full N=128 hd64"), (1, 1, 256, 1, 64, False, "full N=256 hd64"),
                                              (1, 1, 128, 1, 72, False, "full N=128 hd72"), (1, 16, 8, 1, 64, True, "temporal F=16 hd64")]:
        T, D = b * f * n, h * hd
        base = torch.randn(T, 3 * D, generator=g).to(dev).to(dt)
        # (1) V = 1 -> out = 1 whatever S is
        q = base.clone(); q[:, 2 * D:] = 1
        stat(f"attn probe V=1 [{label}]", ops.attention(q, b, f, n, h, temporal), attn_ref(q, b, f, n, h, temporal), 2e-3)
        # (2) Q = 0 -> uniform P -> out = mean_k V : tests the V (MN-major) operand alone
        q = base.clone(); q[:, :D] = 0
        bad = stat(f"attn probe Q=0 [{label}]", ops.attention(q, b, f, n, h, temporal), attn_ref(q, b, f, n, h, temporal), 2e-3)
        if bad.any():
            print("   bad per hd column:", bad.float().mean(0).cpu().numpy().round(2)[:hd])
        # (3) random
        bad = stat(f"attn probe random [{label}]", ops.attention(base, b, f, n, h, temporal), attn_ref(base, b, f, n, h, temporal), 4e-3)
        if bad.any():
            print("   bad per hd column:", bad.float().mean(0).cpu().numpy().round(2)[:hd])
            print("   bad per row (first 32):", bad.float().mean(1).cpu().numpy().round(2)[:32])


def stage_attn():
    g = torch.Generator(device="cpu").manual_seed(4)
    cases = [(2, 16, 256, 6, 64, False), (2, 16, 256, 16, 72, False), (2, 4, 64, 8, 72, False), (3, 8, 64, 2, 64, False),
             (2, 16, 256, 16, 72, True), (2, 16, 256, 6, 64, True), (2, 8, 64, 2, 64, True), (4, 4, 64, 8, 72, True), (1, 2, 16, 2, 64, False)]
    for (b, f, n, h, hd, temporal) in cases:
        for dt in (torch.float16, torch.bfloat16):
            qkv = (torch.randn(b * f * n, 3 * h * hd, generator=g) * 1.5).to(dev).to(dt)
            try:
                out = ops.attention(qkv, b, f, n, h, temporal)
            except RuntimeError as e:
                print(f"[ERR] attn b{b} f{f} n{n} h{h} hd{hd} temporal={temporal}: {e}")
                continue
            stat(f"attn b{b} f{f} n{n} h{h} hd{hd} {'temporal' if temporal else 'spatial'} {str(dt)[6:]}", out,
                 attn_ref(qkv, b, f, n, h, temporal), 4e-3 if dt == torch.float16 else 3e-2)


def _model_case(fname, dtype, also_cfg=True):
    import re
    from oracle import latte_oracle as O
    from latte_b200 import Latte
    gd = np.load(os.path.join(os.path.dirname(OUT), "tests", "golden", fname))
    m = re.match(r"(\S+) batch=(\d+) wseed=(\d+) iseed=(\d+) extras=(\d+) frames=(\d+) input=(\d+)", str(gd["meta"]))
    name, batch, wseed, iseed, extras, frames, inp = m.group(1), *map(int, m.groups()[1:])
    cfg = O.make_config(name, extras=extras, num_frames=frames, input_size=inp)
    sd = O.make_weights(cfg, wseed)
    x, t, y = O.make_inputs(cfg, batch, iseed)
    net = Latte(input_size=cfg.input_size, patch_size=2, in_channels=4, hidden_size=cfg.hidden_size, depth=cfg.depth,
                num_heads=cfg.num_heads, num_frames=cfg.num_frames, num_classes=cfg.num_classes, learn_sigma=True, extras=cfg.extras)
    net.load_state_dict(sd, strict=True)
    net = net.to(dev).eval()
    net.compute_dtype = dtype
    with torch.no_grad():
        out = net(x.to(dev), t.to(dev), y=y.to(dev) if extras == 2 else None)
        torch.cuda.synchronize()
        from oracle import golden as G
        got, ref = G.pair(gd, "out", out)
        stat(f"model {name} {str(dtype)[6:]} vs reference golden (ref's own bf16 dev {float(gd['ref_bf16_maxabs']):.2e})", got, ref.to(dev), 1e-2)
        if also_cfg:
            oc = net.forward_with_cfg(x.to(dev), t.to(dev), y=y.to(dev) if extras == 2 else None, cfg_scale=7.0)
            stat(f"model {name} {str(dtype)[6:]} forward_with_cfg half eps", oc[: batch // 2, :, :4], torch.from_numpy(gd["out_cfg_half_eps"]).to(dev), 6e-2)
    return net, (x, t, y)


def stage_model():
    for fname in ("latte_tiny64_2_b2.npz", "latte_tiny72_2_b2.npz", "latte_tiny72_2_extras1_b4.npz", "latte_s_2_b2.npz"):
        for dt in (torch.float16, torch.bfloat16):
            try:
                _model_case(fname, dt)
            except Exception as e:  # noqa: BLE001
                print(f"[ERR] {fname} {dt}: {type(e).__name__}: {e}")


def stage_xl():
    for dt in (torch.float16, torch.bfloat16):
        net, (x, t, y) = _model_case("latte_xl_2_b2.npz", dt)
        xd, td, yd = x.to(dev), t.to(dev), y.to(dev)
        with torch.no_grad():
            for _ in range(3):
                net.forward_with_cfg(xd, td, y=yd, cfg_scale=7.0)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(10):
                net.forward_with_cfg(xd, td, y=yd, cfg_scale=7.0)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / 10
            print(f"XL/2 B=2 {dt}: {ms:.3f} ms/step  -> {7.451 / ms:.1f} TFLOP/s-equivalent... ({1000 / ms:.1f} steps/s)", flush=True)
        del net


if __name__ == "__main__":
    t0 = time.time()
    print(torch.cuda.get_device_name(0), torch.cuda.get_device_capability(0), flush=True)
    {"ln": stage_ln, "gemm_probe": stage_gemm_probe, "gemm": stage_gemm, "attn_probe": stage_attn_probe,
     "attn": stage_attn, "model": stage_model, "xl": stage_xl}[sys.argv[1]]()
    torch.cuda.synchronize()
    print(f"stage {sys.argv[1]} done in {time.time() - t0:.1f}s", flush=True)

"""bench.py — denoising-steps/sec of the Latte hot path (BASELINE.json metric) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dtype fp16|bf16] [--model Latte-XL/2]
                    [--dump-outputs DIR]

A "step" is one denoising step of `sample/sample.py`: ONE `forward_with_cfg` call on the CFG pair of a
16x(4x32x32) latent video (B_model = 2) — BASELINE.json configs[1], Latte-XL/2 class-conditional 16x256x256.
Synthetic latents, seeded synthetic weights (no checkpoints offline).  Under torchrun (N > 1) every rank is an
independent replica with its own video (sample_ddp.py partitioning): weak scaling, no data-path collective;
`value` = N * K / max-over-ranks device time.

JSON keys beyond the base contract:
  roofline     dominant kernel = the tcgen05 GEMM family (4 launches per block): algorithmic GEMM FLOPs per step /
               summed GEMM device time of a step, measured with CUDA events recorded on the launching stream by the
               library's profiling hook in a SECOND instrumented pass of K steps (the headline pass records nothing)
  cpu_baseline the oracle port (oracle/latte_oracle.py, torch CPU fp32) timed on this box's host cores, rank 0, N=1
  e2e          same metric through the public module call with HOST pinned buffers: H2D of x, forward, D2H of the result
  --impl reference: times the CPU oracle port only (the reference is pure Python and cannot travel; its restatement can).

--dump-outputs DIR writes what the timed step returned in its last timed call as float32 DIR/<name>.npy (rank 0 only):
forward_with_cfg.npy for the Latte workload (both impls, same seeded weights and inputs, so the native and reference
outputs compare directly), t2v_forward.npy for --workload t2v.  Inputs are seeded, so two builds compare output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import datetime
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "denoising-steps/sec Latte-XL/2 16x256x256 (CFG pair per step)"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(tensor_burst=d["bf16_tflops"], tensor_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    hbm=d["hbm_gbs"], source="measured (MEASURED_PEAKS.json)")
    return dict(tensor_burst=1590.0, tensor_sustained=1400.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines, self.t0, self.t1 = index, None, [], None, None

    def start(self):
        """Launch the poller EARLY (before warm-up: nvidia-smi can take a second to come up); only samples whose own
        timestamp falls between mark_begin() and mark_end() are reported."""
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True)
            self.t.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def mark_begin(self):
        self.t0 = datetime.datetime.now()

    def mark_end(self):
        self.t1 = datetime.datetime.now()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)            # let the sample that covers the end of the window arrive
        self.proc.terminate()
        self.t.join(timeout=2)
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f")
                if self.t0 is not None and not (self.t0 <= ts <= (self.t1 or datetime.datetime.now())):
                    continue
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons),
                "window": "device-timed region of `value` + of `e2e` (same workload, back to back)"}


def build_case(model_name: str, seed: int):
    from oracle import latte_oracle as O  # weights/inputs builder + FLOP model only (test infrastructure, not compute)
    cfg = O.make_config(model_name)
    sd = O.make_weights(cfg, 0)
    x, t, y = O.make_inputs(cfg, 2, 123 + seed)
    return O, cfg, sd, x, t, y


def cpu_step_factory(O, model_name, cfg, sd, x, t, y):
    """One `forward_with_cfg` step on the host cores: the UNMODIFIED reference module when oracle/_ref was materialised
    (oracle/make_ref.py), else the oracle port.  Returns (callable, kind, description)."""
    from oracle import ref_loader
    m = ref_loader.build_latte(model_name, cfg, sd)
    if m is not None:
        return (lambda: m.forward_with_cfg(x, t, y=y, cfg_scale=7.0)), "reference", \
            "unmodified reference models/latte.py (oracle/_ref + timm shim), torch CPU fp32 eager, 'math' attention"
    return (lambda: O.latte_forward_with_cfg(sd, cfg, x, t, y, 7.0)), "port", \
        "oracle port of the pure-Python reference (oracle/_ref absent), torch CPU fp32 eager"


def tune_cpu_threads(O, model_name) -> int:
    """torch CPU eager is far from monotone in thread count on many-core hosts (128 threads were 4x slower than 8 on the
    r01 box).  Sweep on the WORKLOAD'S OWN op shapes -- a 2-block model of the same width / heads / token count as
    `model_name` (every Linear, attention and LayerNorm call has the shape it has in the full model; only the block count
    differs) -- and keep the best, so the CPU arm is the reference's best."""
    import dataclasses
    cores = os.cpu_count() or 1
    cfg = dataclasses.replace(O.make_config(model_name), depth=2)
    sd = O.make_weights(cfg, 0)
    x, t, y = O.make_inputs(cfg, 2, 1)
    best, best_t = 1, float("inf")
    for n in sorted({c for c in (8, 16, 32, 64, cores) if c <= cores}):
        torch.set_num_threads(n)
        with torch.no_grad():
            O.latte_forward_with_cfg(sd, cfg, x, t, y, 7.0)          # warm the pool
            t0 = time.perf_counter()
            O.latte_forward_with_cfg(sd, cfg, x, t, y, 7.0)
            el = time.perf_counter() - t0
        if el < best_t:
            best, best_t = n, el
    torch.set_num_threads(best)
    return best


def dump_outputs(directory, arrays: dict) -> None:
    """Write each tensor of `arrays` as float32 `directory/<name>.npy` (bench.py --dump-outputs)."""
    if not directory:
        return
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, f"{name}.npy"), a.detach().float().cpu().numpy())


WORKLOAD = ("{model} class-conditional 16x256x256 sampling step: forward_with_cfg on B_model=2 (1 video x CFG pair) per GPU; "
            "seeded synthetic weights/latents")


def run_reference(args):
    """Reference arm: the reference's own CPU implementation of the step on this box's host cores (rank 0 only): W warm-up
    and exactly K timed `forward_with_cfg` calls, as the main arm."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    O, cfg, sd, x, t, y = build_case(args.model, 0)
    cores = tune_cpu_threads(O, args.model)
    step, kind, what = cpu_step_factory(O, args.model, cfg, sd, x, t, y)
    W, K = max(args.warmup, 0), args.steps
    with torch.no_grad():
        for _ in range(W):
            step()
        t1 = time.perf_counter()
        for _ in range(K):
            out = step()
        el = time.perf_counter() - t1
    dump_outputs(args.dump_outputs, {"forward_with_cfg": out})
    v = K / el
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "steps/s", "n_gpus": args.gpus, "steps": K,
        "warmup": W, "ms_per_step": 1000 * el / K, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD.format(model=args.model)},
        "cpu_baseline": {"value": v, "unit": "steps/s", "cores": cores, "kind": kind,
                         "sample": f"{K} full forward_with_cfg step(s): {what}; {cores} threads = best of a sweep on "
                                   f"{os.cpu_count()} host threads over the model's own op shapes"},
        "e2e": {"value": v, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


def run_t2v(args):
    """Secondary workload (BASELINE configs[3]): one LatteT2V denoising step at 16x512x512, CFG pair (B_model = 2), 120
    synthetic T5 tokens, seeded synthetic weights; then the AutoencoderKLTemporalDecoder decode of the 16 latents in the
    pipeline's chunks of 14 + 2 frames (pipeline_latte.py:785-792).  Prints one JSON line; not the round's bench line."""
    import ctypes as C
    from latte_b200 import LatteT2V, _lib
    from oracle import t2v_oracle as T
    dev = torch.device("cuda", 0)
    lib = _lib.load()
    cfg = T.T2VConfig()
    net = LatteT2V()
    g = torch.Generator().manual_seed(0)
    with torch.no_grad():
        for prm in net.parameters():
            prm.copy_(torch.randn(prm.shape, generator=g) * (0.05 if prm.dim() == 1 else 1.0 / prm.shape[-1] ** 0.5))
    net = net.to(dev).half().eval()
    x, t, text = T.make_inputs(cfg, 2, 120, 1)
    xd, td, txd = x.to(dev), t.to(dev), text.to(dev)
    W, K = max(args.warmup, 3), args.steps
    with torch.no_grad():
        for _ in range(W):
            net(xd, td, encoder_hidden_states=txd, return_dict=False)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(K):
            out = net(xd, td, encoder_hidden_states=txd, return_dict=False)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / K
        dump_outputs(args.dump_outputs, {"t2v_forward": out[0]})
        _lib.profile_enable(True)
        for _ in range(K):
            net(xd, td, encoder_hidden_states=txd, return_dict=False)
        torch.cuda.synchronize()
        pm, pn = (C.c_double * 4)(), (C.c_int * 4)()
        _lib.check(lib.b200_profile_collect(pm, pn, 4), "b200_profile_collect")
        _lib.profile_enable(False)
    peaks = load_peaks()
    fl = 2 * T.algorithmic_flops_per_video(cfg, 120)
    gfl = 2 * T.gemm_flops_per_video(cfg, 120)
    achieved = gfl / (pm[0] / K * 1e-3) / 1e12
    res = {"metric": "denoising-steps/sec LatteT2V 16x512x512 (CFG pair per step)", "value": 1000.0 / ms, "unit": "steps/s",
           "n_gpus": 1, "steps": K, "warmup": W, "ms_per_step": ms, "higher_is_better": True, "dtype": "fp16", "data": "synthetic",
           "config": {"workload": "LatteT2V (Latte-1 config) 16x512x512, B_model=2, 120 text tokens",
                      "algorithmic_tflop_per_step": fl / 1e12, "step_tflops_achieved": fl / (ms * 1e-3) / 1e12},
           "gpu_launches": int(sum(pn) // K),
           "roofline": {"bound": "tensor", "kernel": "gemm_kernel<BN,EPI> (tcgen05)", "achieved": achieved, "peak": peaks["tensor_sustained"],
                        "unit": "TFLOP/s", "frac": achieved / peaks["tensor_sustained"], "traffic": None,
                        "peak_source": peaks["source"] + ", sustained figure", "gemm_ms_per_step": pm[0] / K,
                        "attn_ms_per_step": pm[1] / K, "ln_ms_per_step": pm[2] / K, "other_ms_per_step": pm[3] / K}}
    try:
        from latte_b200 import AutoencoderKLTemporalDecoder
        vae = AutoencoderKLTemporalDecoder().to(dev).half().eval()
        z = torch.randn(16, 4, 64, 64, device=dev)

        def decode():
            with torch.no_grad():
                return torch.cat([vae.decode(z[:14], num_frames=14).sample, vae.decode(z[14:], num_frames=2).sample])
        decode()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(3):
            img = decode()
        e1.record()
        torch.cuda.synchronize()
        ms_dec = e0.elapsed_time(e1) / 3
        res["temporal_decoder"] = {"ms_16_frames_512px": ms_dec, "chunks": "14 + 2 frames (pipeline_latte.py:785-792)",
                                   "tflops_achieved": 16 * 3.043 / (ms_dec * 1e-3), "frac_of_sustained_peak": 16 * 3.043 / (ms_dec * 1e-3) / peaks["tensor_sustained"],
                                   "decoded_shape": list(img.shape)}
    except Exception as e:  # noqa: BLE001
        res["temporal_decoder"] = {"error": repr(e)[:300]}
    print(json.dumps(res), flush=True)


def run_video_leg(net, cfg, xd, yd, dev, world, barrier, sharding):
    """frames/s END TO END (second half of BASELINE.json's metric), measured on every rank: one 16-frame video per rank =
    create_diffusion("250").ddim_sample_loop(model.forward_with_cfg, ...) (sample.py:100-107 on this repo's module and
    fused sampler step) + AutoencoderKL.decode (SD-VAE topology, synthetic weights) + uint8 conversion, then the decoded
    frames of all ranks are gathered with NCCL (sharding.gather_frames: the ONE collective of the sampling path).
    Wall clock incl. host code, max over ranks; value = world * frames / that."""
    from latte_b200 import AutoencoderKL, ops
    from latte_b200.diffusion import create_diffusion
    vae = AutoencoderKL().to(dev).half().eval()
    n_steps = 250
    diffusion = create_diffusion(str(n_steps))
    zz = torch.cat([xd[:1], xd[:1]], 0)
    kw = dict(y=yd, cfg_scale=7.0)

    def one_video():
        with torch.no_grad():
            smp = diffusion.ddim_sample_loop(net.forward_with_cfg, zz.shape, zz, clip_denoised=False, model_kwargs=kw, device=dev)
            smp, _ = smp.chunk(2, dim=0)
            img = vae.decode(smp[0] / 0.18215).sample                                   # (16, 3, 256, 256)
            u8 = ops.frames_to_uint8(img.contiguous(), "sample")                            # sample.py:122, fused with the permute
            return sharding.gather_frames(u8[None])                                       # [world, 16, 256, 256, 3]

    one_video()                     # warm-up: graph capture, VAE packing, NCCL channel setup
    with torch.no_grad():
        zl = smp_latents = torch.randn(cfg.num_frames, 4, cfg.input_size, cfg.input_size, device=dev)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(3):
            vae.decode(zl / 0.18215)
        e1.record()
        torch.cuda.synchronize()
    ms_dec = e0.elapsed_time(e1) / 3
    barrier()
    t0 = time.perf_counter()
    frames = one_video()
    torch.cuda.synchronize()
    sec = sharding.max_over_ranks(time.perf_counter() - t0, dev)
    del smp_latents
    return {"value": world * cfg.num_frames / sec, "unit": "frames/s", "n_gpus": world, "ddim_steps": n_steps,
            "measured": "wall clock (max over ranks) of ddim_sample_loop(250 steps, fused sampler step, trajectory conditioning, graph replay) "
                        "+ AutoencoderKL.decode + uint8 conversion + NCCL all_gather of the decoded frames; one 16-frame video per GPU",
            "sec_per_video": sec, "ms_per_step_incl_sampler": (sec * 1e3 - ms_dec) / n_steps, "vae_decode_ms_16_frames": ms_dec,
            "vae_tflops_achieved": 16 * 0.622 / (ms_dec * 1e-3), "gathered_shape": list(frames.shape),
            "gather_bytes_per_rank": int(frames.numel() // world)}


def run_ddp_batch_leg(net, cfg, args, dev, world, rank, barrier, sharding, steps):
    """BASELINE configs[2]: the sample_ddp.py batch -- per_proc_batch_size 2 videos per rank (ucf101_sample.yaml), i.e.
    B_model = 4 rows per forward_with_cfg -- as device-timed steps/s (one step advances 2 videos per GPU)."""
    from oracle import latte_oracle as O
    x4, t4, y4 = O.make_inputs(cfg, 4, 777 + sharding.rank_seed(0, rank, world))
    x4, t4, y4 = x4.to(dev), t4.to(dev), y4.to(dev)
    with torch.no_grad():
        for _ in range(3):
            net.forward_with_cfg(x4, t4, y=y4, cfg_scale=7.0)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(steps):
            net.forward_with_cfg(x4, t4, y=y4, cfg_scale=7.0)
        e1.record()
        barrier()
    ms = sharding.max_over_ranks(e0.elapsed_time(e1), dev) / steps
    return {"value": world * 1000.0 / ms, "unit": "steps/s (B_model = 4: 2 videos x CFG pair per GPU per step)", "ms_per_step": ms,
            "steps": steps, "videos_per_step": 2 * world}


def run_train_leg(args, dev, world, rank, barrier, sharding, steps=5, local_batch=5):
    """BASELINE configs[4] (SURVEY 8d config 5): Latte-XL/2 training step as train.py:206-222 runs it -- fp32 parameters,
    `torch.autocast(bfloat16)`, `diffusion.training_losses` (MSE + VB), `loss.backward()` -- local batch 5 of synthetic
    latents (VAE encode skipped, as the config says), DistributedDataParallel gradient all-reduce at N > 1.  Metric: fwd+bwd
    steps/s (no optimizer step, per the config).  At N = 1 the UNMODIFIED reference module is timed the same way on this GPU."""
    import torch.distributed as dist
    from latte_b200 import Latte_models
    from latte_b200.diffusion import create_diffusion
    torch.manual_seed(1234 + rank)
    try:
        with torch.device(dev):                             # parameters are created and initialised on the GPU (674 M of them)
            model = Latte_models[args.model](input_size=32, num_classes=101, num_frames=16, learn_sigma=True, extras=2)
    except Exception:  # noqa: BLE001  (a torch build without device-context factories): build on the host, then move
        model = Latte_models[args.model](input_size=32, num_classes=101, num_frames=16, learn_sigma=True, extras=2).to(dev)
    assert model.pos_embed.device == dev
    with torch.no_grad():
        zero_init = [b.adaLN_modulation[1] for b in model.blocks] + [model.final_layer.adaLN_modulation[1], model.final_layer.linear]
        for lin in zero_init:                              # adaLN-Zero / final layer start at zero: give every parameter a gradient
            lin.weight.normal_(0, 0.02)
            lin.bias.normal_(0, 0.02)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()} if world == 1 else None
    model.train()
    net = torch.nn.parallel.DistributedDataParallel(model, device_ids=[dev.index]) if world > 1 else model
    diffusion = create_diffusion(timestep_respacing="")
    x = torch.randn(local_batch, 16, 4, 32, 32, device=dev)
    y = torch.randint(0, 101, (local_batch,), device=dev)

    def step(module, diff):
        t = torch.randint(0, diff.num_timesteps, (local_batch,), device=dev)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            loss = diff.training_losses(module, x, t, dict(y=y))["loss"].mean()
        module.zero_grad(set_to_none=True)
        loss.backward()
        return loss

    def timed(module, diff, n):
        for _ in range(2):
            step(module, diff)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(n):
            loss = step(module, diff)
        e1.record()
        barrier()
        return sharding.max_over_ranks(e0.elapsed_time(e1), dev) / n, float(loss.detach())

    ms, loss = timed(net, diffusion, steps)
    flops = 3.0 * 3.7256e12 * local_batch                  # fwd + 2x for dgrad/wgrad, SURVEY App. A per-video forward FLOPs
    res = {"value": world * 1000.0 / ms, "unit": "fwd+bwd steps/s (local batch 5 per GPU)", "ms_per_step": ms, "steps": steps,
           "local_batch": local_batch, "global_batch": local_batch * world, "dtype": "bf16 operands, fp32 master parameters / gradients",
           "loss": loss, "algorithmic_tflops_achieved": flops / (ms * 1e-3) / 1e12,
           "peak_mem_gb": torch.cuda.max_memory_allocated(dev) / 2 ** 30,
           "grad_sync": "DistributedDataParallel (NCCL all-reduce, bucketed, overlapped with the backward)" if world > 1 else "none (1 GPU)"}
    del net, model
    torch.cuda.empty_cache()
    if world == 1:
        try:
            from oracle import ref_loader
            import types
            ref_model = ref_loader.build_latte(args.model, types.SimpleNamespace(input_size=32, num_classes=101, num_frames=16,
                                                                                  learn_sigma=True, extras=2), sd)
            if ref_model is not None:
                ref_model = ref_model.to(dev).train()
                ref_diffusion = ref_loader.load_diffusion().create_diffusion(timestep_respacing="")
                torch.backends.cuda.matmul.allow_tf32 = True
                torch.backends.cudnn.allow_tf32 = True
                ms_ref, loss_ref = timed(ref_model, ref_diffusion, max(2, steps // 2))
                res["gpu_eager_baseline"] = {"value": 1000.0 / ms_ref, "unit": "fwd+bwd steps/s", "ms_per_step": ms_ref, "loss": loss_ref,
                                             "kind": "reference (unmodified models/latte.py + diffusion/ from oracle/_ref, PyTorch eager "
                                                     "autograd under bf16 autocast on this GPU, as train.py runs it)",
                                             "speedup": ms_ref / ms}
                del ref_model
            else:
                res["gpu_eager_baseline"] = {"unavailable": "oracle/_ref not present on this box"}
        except Exception as e:  # noqa: BLE001
            res["gpu_eager_baseline"] = {"error": repr(e)[:300]}
        torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--dtype", default="fp16", choices=["fp16", "bf16"])
    ap.add_argument("--model", default="Latte-XL/2")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-video", action="store_true", help="skip the measured 250-step video + VAE decode (profiler runs)")
    ap.add_argument("--workload", default="latte", choices=["latte", "t2v"],
                    help="latte = BASELINE configs[1] (the bench line); t2v = configs[3] denoiser step, a secondary measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the output of the last timed step as float32 DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.workload == "t2v":
        return run_t2v(args)
    if args.impl == "reference":
        return run_reference(args)

    import torch.distributed as dist
    from latte_b200 import Latte, _lib, sharding

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    W, K = max(args.warmup, 3), args.steps

    O, cfg, sd, x, t, y = build_case(args.model, sharding.rank_seed(0, rank, world))
    net = Latte(input_size=cfg.input_size, hidden_size=cfg.hidden_size, depth=cfg.depth, num_heads=cfg.num_heads,
                num_frames=cfg.num_frames, num_classes=cfg.num_classes, learn_sigma=True, extras=2)
    net.load_state_dict(sd, strict=True)
    net = net.to(dev).eval()
    net.compute_dtype = torch.float16 if args.dtype == "fp16" else torch.bfloat16
    lib = _lib.load()
    xd, td, yd = x.to(dev), t.to(dev), y.to(dev)
    x_host = x.clone().pin_memory()
    out_host = [torch.empty(2, cfg.num_frames, cfg.out_channels, cfg.input_size, cfg.input_size).pin_memory() for _ in range(2)]
    out_ready = [torch.cuda.Event(), torch.cuda.Event()]
    e2e_count = [0]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_resident():
        return net.forward_with_cfg(xd, td, y=yd, cfg_scale=7.0)

    def step_e2e():
        """One step as a serving loop issues it: H2D of this step's latents from pinned memory, the public module call, D2H of
        the result into one of two pinned buffers.  The host waits for a buffer only when it is about to be reused (two steps
        later), so enqueueing step i+1 overlaps the GPU work of step i; every result still lands in host memory inside the
        timed region (the closing barrier + synchronize waits for the last two)."""
        k = e2e_count[0] & 1
        e2e_count[0] += 1
        out_ready[k].synchronize()           # the result this buffer held two steps ago is on the host: safe to overwrite
        xg = x_host.to(dev, non_blocking=True)
        o = net.forward_with_cfg(xg, td, y=yd, cfg_scale=7.0)
        out_host[k].copy_(o, non_blocking=True)
        out_ready[k].record()

    last = {}

    def timed(fn, n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(n):
            last["out"] = fn()
        e1.record()
        barrier()
        return sharding.max_over_ranks(e0.elapsed_time(e1), dev)

    with torch.no_grad():
        clocks = ClockSampler(local)
        if rank == 0:
            clocks.start()
        for _ in range(W):
            step_resident()
        for _ in range(2):
            step_e2e()
        clocks.mark_begin()
        ms_total = timed(step_resident, K)
        resident_out = last["out"]
        ms_e2e = timed(step_e2e, K)
        clocks.mark_end()
        clk = clocks.stop() if rank == 0 else None
        # the same step over 250 back-to-back calls (one DDIM-250 video's worth): the power-capped, sustained-clock figure
        ms_sustained = timed(step_resident, 250) / 250

        # instrumented pass: per-kernel-class device time from events on the launching stream
        import ctypes as C
        _lib.profile_enable(True)       # the modules launch eagerly (no graph replay) while events bracket every kernel
        barrier()
        for _ in range(K):
            step_resident()
        torch.cuda.synchronize()
        ms = (C.c_double * 4)()
        nl = (C.c_int * 4)()
        _lib.check(lib.b200_profile_collect(ms, nl, 4), "b200_profile_collect")
        _lib.profile_enable(False)
    if rank == 0:
        dump_outputs(args.dump_outputs, {"forward_with_cfg": resident_out})

    # ---- legs every rank takes part in (they end in a collective): frames/s end to end and the sample_ddp batch
    video_leg, ddp_leg, train_leg = None, None, None
    if not args.no_video:
        try:
            video_leg = run_video_leg(net, cfg, xd, yd, dev, world, barrier, sharding)
        except Exception as e:  # noqa: BLE001
            video_leg = {"error": repr(e)[:300]}
        try:
            ddp_leg = run_ddp_batch_leg(net, cfg, args, dev, world, rank, barrier, sharding, max(K // 2, 5))
        except Exception as e:  # noqa: BLE001
            ddp_leg = {"error": repr(e)[:300]}
        try:
            net._graphs = None                   # release the sampling path's graph scratch before the training leg allocates
            torch.cuda.empty_cache()
            train_leg = run_train_leg(args, dev, world, rank, barrier, sharding)
        except Exception as e:  # noqa: BLE001
            train_leg = {"error": repr(e)[:300]}
    if world > 1:
        dist.barrier()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = load_peaks()
    D, T = cfg.hidden_size, 2 * cfg.num_frames * cfg.num_patches
    gemm_flops_step = 2.0 * T * (D * 3 * D + D * D + 2 * D * int(D * cfg.mlp_ratio)) * cfg.depth  # the 4 Linears of every block
    step_flops = 2 * O.algorithmic_flops_per_video(cfg)
    gemm_ms_step = ms[0] / K
    achieved = gemm_flops_step / (gemm_ms_step * 1e-3) / 1e12
    launches = sum(nl) // K
    # DRAM bytes per GEMM launch from the committed ncu --set full capture (tools/ncu_traffic.py), same units as `achieved`'s
    # numerator is per launch; null until a capture of the current kernels has been committed
    traffic, traffic_src = None, None
    tpath = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "gemm_traffic.json")
    if os.path.exists(tpath):
        with open(tpath) as fh:
            tj = json.load(fh)
        traffic, traffic_src = tj.get("dram_bytes_per_launch"), tj.get("source")
    res = {
        "metric": METRIC, "value": world * K / (ms_total * 1e-3), "unit": "steps/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": args.dtype, "data": "synthetic",
        "config": {"workload": WORKLOAD.format(model=args.model),
                   "l2": "no explicit flush: 1.35 GB of 16-bit weights stream through the 126 MB L2 every step",
                   "parallelism": f"replicas x{world} (sample_ddp partitioning), no data-path collective",
                   "algorithmic_tflop_per_step": step_flops / 1e12,
                   "step_tflops_achieved": step_flops / (ms_total / K * 1e-3) / 1e12},
        "e2e": {"value": world * K / (ms_e2e * 1e-3), "unit": "steps/s", "h2d_bytes_per_step": x_host.numel() * 4,
                "d2h_bytes_per_step": out_host[0].numel() * 4,
                "pattern": "pinned H2D -> Latte.forward_with_cfg (CUDA-graph replay) -> pinned D2H, double-buffered: the host waits on a "
                           "result buffer only before reusing it"},
        "sustained": {"ms_per_step": ms_sustained, "value": world * 1000.0 / ms_sustained, "steps": 250,
                      "note": "same step, 250 back-to-back calls (sustained clocks under the power cap); `value` above is the K-step burst"},
        "gpu_launches": int(launches),
        "roofline": {"bound": "tensor", "kernel": "gemm_kernel<BN,EPI> (tcgen05, 4 launches/block)",
                     "achieved": achieved, "peak": peaks["tensor_sustained"], "unit": "TFLOP/s",
                     "frac": achieved / peaks["tensor_sustained"], "traffic": traffic, "traffic_source": traffic_src,
                     "peak_source": peaks["source"] + ", sustained figure (kernel timed inside a long step)",
                     "gemm_ms_per_step": gemm_ms_step, "attn_ms_per_step": ms[1] / K, "ln_ms_per_step": ms[2] / K,
                     "other_ms_per_step": ms[3] / K, "instrumented_pass_ms_per_step": sum(ms) / K},
        "clocks": clk,
    }
    if video_leg is not None:
        res["frames_per_sec_e2e"] = video_leg
    if ddp_leg is not None:
        res["sample_ddp_batch"] = ddp_leg
    if train_leg is not None:
        res["train_fwd_bwd"] = train_leg
    if world == 1 and not args.no_video:
        # The reference's own 1-GPU path (north_star's ">= 5x" denominator): the UNMODIFIED reference module run as PyTorch
        # eager on this GPU exactly as sample.py does (model.half(), use_fp16=True, tf32 allowed, 'math' attention) when
        # oracle/_ref is present, else the oracle port -- a baseline leg, never part of the product path.
        try:
            from oracle import ref_loader
            torch.backends.cuda.matmul.allow_tf32 = True
            torch.backends.cudnn.allow_tf32 = True
            ref_model = ref_loader.build_latte(args.model, cfg, sd)
            if ref_model is not None:
                ref_model = ref_model.to(dev).half()
                xg = xd.half()
                eager_step = lambda: ref_model.forward_with_cfg(xg, td, y=yd, cfg_scale=7.0, use_fp16=True)   # noqa: E731
                kind = "reference (unmodified models/latte.py from oracle/_ref, PyTorch eager fp16 on this GPU, cuBLAS/ATen kernels)"
            else:
                sdg = {k: v.to(dev).half() for k, v in sd.items()}
                xg = xd.half()
                eager_step = lambda: O.latte_forward_with_cfg(sdg, cfg, xg, td, yd, 7.0, dtype=torch.float16)   # noqa: E731
                kind = "port (oracle restatement, PyTorch eager fp16 on this GPU, cuBLAS/ATen kernels)"
            with torch.no_grad():
                for _ in range(max(W, 3)):
                    eager_step()
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(K):
                    eager_step()
                e1.record()
                torch.cuda.synchronize()
            ms_eager = e0.elapsed_time(e1) / K
            res["gpu_eager_baseline"] = {"value": 1000.0 / ms_eager, "unit": "steps/s", "ms_per_step": ms_eager, "steps": K,
                                         "kind": kind, "speedup_of_value": (K / (ms_total * 1e-3)) / (1000.0 / ms_eager),
                                         "speedup_of_e2e": (K / (ms_e2e * 1e-3)) / (1000.0 / ms_eager)}
            del ref_model
        except Exception as e:  # noqa: BLE001
            res["gpu_eager_baseline"] = {"error": repr(e)[:200]}
    if not args.no_cpu_baseline and world == 1:
        cores = tune_cpu_threads(O, args.model)
        step, kind, what = cpu_step_factory(O, args.model, cfg, sd, x, t, y)
        with torch.no_grad():
            t0 = time.perf_counter()
            step()
            el = time.perf_counter() - t0
        res["cpu_baseline"] = {"value": 1.0 / el, "unit": "steps/s", "cores": cores, "kind": kind,
                               "sample": f"1 full forward_with_cfg step: {what}; {cores} threads = best of a sweep on "
                                         f"{os.cpu_count()} host threads over the model's own op shapes"}
    else:
        res["cpu_baseline"] = None
    print(json.dumps(res), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

"""Throughput at I2VGen-XL's native frame size: 16 frames at 1280 x 704 (latent 160 x 88) and at 704 x 1280, through the product
pipeline with CUDA graphs — the 50 + 50-step job of bench.py (seeded synthetic conditioning, random-init full-size UNet, headline
injection schedule pnp_f_t = pnp_spatial_attn_t = 1.0, cfg 9) at the other frame sizes.

    python tools/native_resolution_bench.py [--steps 3] [--warmup 2] [--out FILE]

Prints one JSON line per frame size (ms per inversion / edit step, steps/s of the 50 + 50 job, peak memory), one line with the
finest-level resnet convolution (48 frames x 160 x 88, 320 -> 320) against the same convolution at the 512 x 512 geometry (48 x
64 x 64) in output pixels/s, and the GPU name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time
from types import SimpleNamespace

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

N_SCHEDULE = 50
GUIDANCE = 9.0
PNP = dict(pnp_f_t=1.0, pnp_spatial_attn_t=1.0, pnp_temp_attn_t=0.0)


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in q.split(",")]
    except Exception:  # noqa: BLE001 - the numbers are still printed; the line says what could not be read
        name, power = torch.cuda.get_device_name(), "unknown"
    return {"gpu": name, "power_limit": power}


def time_job(pipe, frames, h, w, steps, warmup, dev):
    from anyv2v_b200.latent_store import LatentStore
    from anyv2v_b200.run_group_pnp_edit import init_pnp, synthetic_conditioning
    from anyv2v_b200.schedulers import DDIMInverseScheduler, DDIMScheduler
    cond = {k: v.to(dev) for k, v in synthetic_conditioning(frames, h, w, 1024, 8888, "cpu").items()}
    torch.cuda.reset_peak_memory_stats(dev)
    pipe.scheduler = inv_sched = DDIMInverseScheduler()
    st_inv = pipe.prepare_invert(cond["video_latents"], cond["inv_prompt"], cond["src_image_latents"], cond["src_image_emb"], 8,
                                 N_SCHEDULE, 1.0, None, False, False)
    edit_sched = DDIMScheduler()
    edit_sched.set_timesteps(N_SCHEDULE)
    pipe.scheduler = edit_sched
    init_pnp(pipe, edit_sched, SimpleNamespace(n_steps=N_SCHEDULE, **PNP))
    # the edit loop reads x_t of the source for t = 981, 961, ...: a short run pre-seeds the store with seeded latents for them
    store = LatentStore(None, write_files=False)
    g = torch.Generator().manual_seed(4242)
    for t in edit_sched.timesteps.tolist()[:steps + warmup]:
        store._mem[int(t)] = torch.randn(1, 4, frames, h, w, generator=g).half().to(dev)
    st_edit = pipe.prepare_edit(cond["video_latents"].clone(), cond["edit_prompt"], cond["neg_prompt"], cond["inv_prompt"],
                                cond["edit_image_emb"], cond["edit_image_latents"], cond["src_image_emb"], cond["src_image_latents"],
                                8, N_SCHEDULE, GUIDANCE, 0, None, store, True)
    st_inv.store = store

    def phase(step, st, sched, i0, n):
        pipe.scheduler = sched
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(i0, i0 + n):
            step(st, i)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / max(n, 1)

    phase(pipe.invert_step, st_inv, inv_sched, 0, warmup)  # eager pass, then CUDA-graph capture
    phase(pipe.edit_step, st_edit, edit_sched, 0, warmup)
    ms_inv = phase(pipe.invert_step, st_inv, inv_sched, warmup, steps)
    ms_edit = phase(pipe.edit_step, st_edit, edit_sched, warmup, steps)
    finite = bool(torch.isfinite(st_inv.latents).all() and torch.isfinite(st_edit.latents).all())
    job_s = N_SCHEDULE * (ms_inv + ms_edit) * 1e-3
    return {"ms_per_inversion_step": round(ms_inv, 2), "ms_per_edit_step": round(ms_edit, 2),
            "steps_per_s_50_plus_50": round(2 * N_SCHEDULE / job_s, 4), "job_s": round(job_s, 2),
            "peak_memory_gb": round(torch.cuda.max_memory_allocated(dev) / 2 ** 30, 2), "outputs_finite": finite}


def time_conv(ops, nf, h, w, c, dev, iters=20):
    """the finest-level resnet convs: conv1 (+ time-embedding row bias) and conv2 (+ shortcut residual), output pixels/s"""
    g = torch.Generator(device=dev).manual_seed(5)
    x = torch.randn(nf, h, w, c, device=dev, generator=g).half()
    wt = (torch.randn(c, 9 * c, device=dev, generator=g) / (9 * c) ** 0.5).half()
    b = torch.randn(c, device=dev, generator=g).half()
    temb = torch.randn(nf, c, device=dev, generator=g).half()
    res = torch.randn(nf, h, w, c, device=dev, generator=g).half()
    out = torch.empty(nf, h, w, c, device=dev, dtype=torch.float16)
    calls = {"conv1_rowbias": lambda: ops.conv3x3(x, wt, bias=b, rowbias=temb, rows_per_rowbias=h * w, out=out),
             "conv2_residual": lambda: ops.conv3x3(x, wt, bias=b, residual=res, out=out)}
    rec = {}
    for name, fn in calls.items():
        for _ in range(3):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) * 1e3 / iters
        rec[name] = {"us": round(us, 2), "gpix_per_s": round(nf * h * w / us * 1e-3, 3),
                     "tflops": round(2.0 * nf * h * w * c * 9 * c / us * 1e-6, 1)}
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=16)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    from anyv2v_b200 import distributed, ops
    from anyv2v_b200.pipeline import I2VGenXLPipeline
    from anyv2v_b200.schedulers import DDIMInverseScheduler
    from anyv2v_b200.unet_i2vgen_xl import I2VGEN_XL_CONFIG, I2VGenXLUNet
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    torch.set_grad_enabled(False)
    info = gpu_info()
    lines = []
    conv = {"latent_160x88": time_conv(ops, 48, 88, 160, 320, dev), "latent_64x64": time_conv(ops, 48, 64, 64, 320, dev)}
    conv["ratio_160x88_over_64x64_pixels_per_s"] = {k: round(conv["latent_160x88"][k]["gpix_per_s"] / conv["latent_64x64"][k]["gpix_per_s"], 3)
                                                    for k in conv["latent_160x88"]}
    lines.append(dict(record="finest-level resnet conv, 48 frames, 320 -> 320 channels (CUDA events, 20 launches)", **conv, **info))
    t0 = time.time()
    unet = distributed.build_unet_replicated(I2VGenXLUNet, I2VGEN_XL_CONFIG, 8888, dev, broadcast=False)  # bench.py's weights
    pipe = I2VGenXLPipeline(unet, DDIMInverseScheduler())
    build_s = time.time() - t0
    for wp, hp in ((1280, 704), (704, 1280)):
        rec = time_job(pipe, args.frames, hp // 8, wp // 8, args.steps, args.warmup, dev)
        lines.append(dict(record=f"{args.frames} frames at {wp}x{hp} (latent {wp // 8}x{hp // 8}), 50 inversion + 50 PnP edit steps, "
                                 f"cfg {GUIDANCE}, pnp {PNP}, CUDA graphs, {args.steps} timed steps per phase after {args.warmup}",
                          **rec, model_build_s=round(build_s, 1), **info))
        torch.cuda.empty_cache()
    for rec in lines:
        s = json.dumps(rec)
        print(s, flush=True)
        if args.out:
            with open(args.out, "a") as fh:
                fh.write(s + "\n")


if __name__ == "__main__":
    main()

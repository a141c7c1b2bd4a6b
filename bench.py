"""Benchmark of the AnyV2V hot path on B200: denoising-steps/sec of I2VGen-XL DDIM inversion + PnP edit.

  python bench.py --gpus N --steps K --warmup W            # this package (CUDA kernels through the C ABI)
  python bench.py --impl reference --gpus N --steps K ...   # the reference path's CPU port (oracle) on the host cores
  python bench.py ... --dump-outputs DIR                    # also write the last timed step's latents to DIR/*.npy

Workload (BASELINE.json configs[1], the configuration the metric is quoted on): one 16-frame 512x512 clip
(latents [1,4,16,64,64]), full-size random-init I2VGen-XL UNet (1.42 B params, fp16), 50-step schedules, guidance 9.0,
conv + spatial-attention injection on every edit step (pnp_f_t = pnp_spatial_attn_t = 1.0, pnp_temp_attn_t = 0), seeded
synthetic conditioning (SURVEY 8d).  One "step" = one denoising step.  The timed K steps are K/2 inversion steps (UNet
batch 1) followed by K/2 PnP-edit steps (UNet batch 3: source / uncond / cond), the 1:1 mix of the 50 + 50 job, taken
from the start of the two 50-step schedules; the edit steps consume the inverted latents the inversion steps produced.
Under torchrun every rank runs its own clip (weak scaling; the only collective is the one-time weight broadcast).

Besides the headline the same line carries (all measured live in this run):
  * ``sub_records.config3`` — BASELINE.json configs[2]: the full conv + spatial + temporal injection schedule (pnp_f_t 0.8,
    pnp_spatial_attn_t = pnp_temp_attn_t = 0.5): per-step times of its three step classes (all hooks / conv only / dead source
    branch) and the 50 + 50-step job throughput they add up to;
  * ``roofline`` — the injected spatial self-attention (tensor-bound), ``roofline_more`` — the fused temporal attention of an
    injected step and GroupNorm+SiLU (both HBM-bound) and two shapes of the GEMM kernel (the dominant kernel by time);
  * ``weights_broadcast`` — the one NCCL collective (ms, GB/s) under torchrun.
``--frames 128`` switches the workload to BASELINE.json configs[4] (128-frame long-video clip per GPU).

One JSON line is printed by rank 0 (see README / the driver contract for the keys).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

F, H, W = 16, 64, 64
N_SCHEDULE = 50
GUIDANCE = 9.0
PNP = dict(pnp_f_t=1.0, pnp_spatial_attn_t=1.0, pnp_temp_attn_t=0.0)          # BASELINE configs[1] (headline)
PNP_CONFIG3 = dict(pnp_f_t=0.8, pnp_spatial_attn_t=0.5, pnp_temp_attn_t=0.5)  # BASELINE configs[2]
PNP_LONG = dict(pnp_f_t=1.0, pnp_spatial_attn_t=1.0, pnp_temp_attn_t=1.0)     # BASELINE configs[4] (--frames 128; gradio rows 0.5-1.0)
METRIC = "denoising-steps/sec (16f x 512^2 I2VGen-XL, 50 inv + 50 edit PnP sampling)"
# algorithmic FLOPs per step of the reference computation (SURVEY Appendix B), 2*MAC
TFLOP_INV, TFLOP_EDIT = 20.94, 62.81


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            d = json.load(fh)
        return dict(source="measured (MEASURED_PEAKS.json)", hbm_gbs=d["hbm_gbs"], tflops_burst=d["bf16_tflops"],
                    tflops_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]))
    return dict(source="fallback (B200_PROFILING.md)", hbm_gbs=6650.0, tflops_burst=1590.0, tflops_sustained=1400.0)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, reasons = [], None, set()
        for l in self.lines:
            p = [x.strip() for x in l.split(",")]
            if len(p) < 8:
                continue
            try:
                sm.append(float(p[1]))
                smax = float(p[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons), "samples": len(sm)}


# =============================================================================================== our arm (GPU)
def synthetic(device, seed, pinned_host=False):
    from anyv2v_b200.run_group_pnp_edit import synthetic_conditioning
    c = synthetic_conditioning(F, H, W, 1024, seed, "cpu")
    if pinned_host:
        return {k: v.pin_memory() for k, v in c.items()}
    return {k: v.to(device) for k, v in c.items()}


def run_ours(args):
    from anyv2v_b200 import distributed, ops
    from anyv2v_b200.pipeline import I2VGenXLPipeline
    from anyv2v_b200.run_group_pnp_edit import init_pnp
    from anyv2v_b200.schedulers import DDIMInverseScheduler, DDIMScheduler
    from anyv2v_b200.unet_i2vgen_xl import I2VGEN_XL_CONFIG, I2VGenXLUNet
    from types import SimpleNamespace

    rank, local, world = distributed.init_from_env()
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    torch.set_grad_enabled(False)
    K, Wm = args.steps, args.warmup
    k_inv, k_edit = (K + 1) // 2, K // 2
    w_inv, w_edit = (Wm + 1) // 2, Wm // 2
    assert k_inv + w_inv <= N_SCHEDULE and k_edit + w_edit <= N_SCHEDULE

    t0 = time.time()
    unet = distributed.build_unet_replicated(I2VGenXLUNet, I2VGEN_XL_CONFIG, 8888, dev)  # rank 0 inits, NCCL broadcast
    torch.cuda.synchronize()
    build_s = time.time() - t0
    pipe = I2VGenXLPipeline(unet, DDIMInverseScheduler())
    edit_sched = DDIMScheduler()
    edit_sched.set_timesteps(N_SCHEDULE)
    pnp = PNP_LONG if F > 16 else PNP
    pnp_cfg = SimpleNamespace(n_steps=N_SCHEDULE, **pnp)
    torch.cuda.reset_peak_memory_stats(dev)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def phase_states(cond, host_resident):
        """prepare both phases; the edit phase reads x_t for t = 981, 961, ... which the inversion phase only produces
        after 50 steps — for a K-step bench the store is pre-seeded with synthetic source latents for those t."""
        pipe.scheduler = inv_sched = DDIMInverseScheduler()
        st_inv = pipe.prepare_invert(cond["video_latents"], cond["inv_prompt"], cond["src_image_latents"], cond["src_image_emb"],
                                     8, N_SCHEDULE, 1.0, None, False, host_resident)
        store = st_inv.store
        pipe.scheduler = edit_sched
        init_pnp(pipe, edit_sched, pnp_cfg)
        st_edit = pipe.prepare_edit(cond["video_latents"].clone(), cond["edit_prompt"], cond["neg_prompt"], cond["inv_prompt"],
                                    cond["edit_image_emb"], cond["edit_image_latents"], cond["src_image_emb"],
                                    cond["src_image_latents"], 8, N_SCHEDULE, GUIDANCE, 0, None, store, True)
        return inv_sched, st_inv, st_edit

    launches_per_step = {}

    def run_steps(inv_sched, st_inv, st_edit, i0_inv, n_inv, i0_edit, n_edit, d2h_result=None):
        pipe.scheduler = inv_sched
        for i in range(i0_inv, i0_inv + n_inv):
            c0 = ops.launch_count()
            x = pipe.invert_step(st_inv, i)
            launches_per_step.setdefault("inv", ops.launch_count() - c0)  # first (eager) pass = launches per step
            if d2h_result is not None:
                d2h_result.copy_(x, non_blocking=True)
        pipe.scheduler = edit_sched
        for i in range(i0_edit, i0_edit + n_edit):
            c0 = ops.launch_count()
            x = pipe.edit_step(st_edit, i)
            launches_per_step.setdefault("edit", ops.launch_count() - c0)
            if d2h_result is not None:
                d2h_result.copy_(x, non_blocking=True)

    # ------------------------------------------------------------------ value: inputs resident in HBM
    from anyv2v_b200.latent_store import LatentStore
    cond_dev = synthetic(dev, 8888 + rank)
    inv_sched, st_inv, st_edit = phase_states(cond_dev, host_resident=False)
    g_seed = torch.Generator().manual_seed(4242 + rank)
    src_latents = {int(t): torch.randn(1, 4, F, H, W, generator=g_seed).half()
                   for t in edit_sched.timesteps.tolist()[: max(k_edit + w_edit, k_edit)]}

    def reset(host_resident):
        """fresh latents + a fresh latent store; the captured CUDA graphs (static buffers) are kept"""
        st_inv.latents.copy_(cond_dev["video_latents"])
        st_edit.latents.copy_(cond_dev["video_latents"])
        store = LatentStore(None, write_files=False, host_resident=host_resident)
        for t, x in src_latents.items():
            store._mem[t] = x.pin_memory() if host_resident else x.to(dev)
        st_inv.store = st_edit.store = store
        return store

    reset(False)
    run_steps(inv_sched, st_inv, st_edit, 0, w_inv, 0, w_edit)  # warm-up: eager pass, then CUDA-graph capture
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = ops.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    run_steps(inv_sched, st_inv, st_edit, w_inv, k_inv, w_edit, k_edit)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    # what the last timed step of each phase returned to its caller, copied before the passes below reuse the static buffers
    last_outputs = {}
    if args.dump_outputs:
        if k_inv:
            last_outputs["inversion_latents"] = st_inv.latents.float().cpu()
        if k_edit:
            last_outputs["edit_latents"] = st_edit.latents.float().cpu()
    graphs = pipe.use_cuda_graphs
    # kernels launched per replayed step are the ones recorded at capture time
    launches = ops.launch_count() - l0
    if graphs:
        launches = int(round(launches_per_step["inv"] * k_inv + launches_per_step["edit"] * k_edit))
    clocks = sampler.stop() if rank == 0 else None
    finite = bool(torch.isfinite(st_edit.latents).all() and torch.isfinite(st_inv.latents).all())
    # per-phase split (not part of the contract): a second, separately timed pass over the same steps
    reset(False)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    torch.cuda.synchronize()
    ev[0].record()
    run_steps(inv_sched, st_inv, st_edit, w_inv, k_inv, 0, 0)
    ev[1].record()
    run_steps(inv_sched, st_inv, st_edit, 0, 0, w_edit, k_edit)
    ev[2].record()
    torch.cuda.synchronize()
    ms_inv, ms_edit = ev[0].elapsed_time(ev[1]) / max(k_inv, 1), ev[1].elapsed_time(ev[2]) / max(k_edit, 1)

    # ------------------------------------------------------------------ rooflines of the hot kernels, in situ
    roof = attention_roofline(ops, dev)
    roof_more = [temporal_attention_roofline(ops, dev), groupnorm_roofline(ops, dev), *gemm_rooflines(ops, dev)]

    # ------------------------------------------------------------------ e2e: host buffers, copies inside the timed region
    cond_host = synthetic(dev, 8888 + rank, pinned_host=True)
    result_host = torch.empty(1, 4, F, H, W, dtype=torch.float16).pin_memory()
    step_io = F * H * W * 4 * 2
    store = reset(True)
    barrier()
    t_start = time.perf_counter()
    for k, v in cond_host.items():  # conditioning + initial latents: pinned host -> device
        cond_dev[k].copy_(v, non_blocking=True)
    st_inv.latents.copy_(cond_dev["video_latents"])
    st_edit.latents.copy_(cond_dev["video_latents"])
    run_steps(inv_sched, st_inv, st_edit, w_inv, k_inv, w_edit, k_edit, d2h_result=result_host)
    torch.cuda.synchronize()
    t_e2e = time.perf_counter() - t_start
    barrier()
    h2d_total = store.h2d_bytes + sum(v.numel() * v.element_size() for v in cond_host.values())
    d2h_total = store.d2h_bytes + K * step_io

    # ------------------------------------------------------------------ BASELINE configs[2]: full injection schedule
    # (after everything that replays the headline graphs: the hook registration is module state read by edit_step)
    sub = {}
    if F == 16:
        sub["config3"] = config3_record(pipe, edit_sched, cond_dev, dev, ms_inv, init_pnp)
        init_pnp(pipe, edit_sched, pnp_cfg)
    peak_mem_gb = torch.cuda.max_memory_allocated(dev) / 2 ** 30

    # ------------------------------------------------------------------ reduce over ranks (max time)
    t = torch.tensor([ms, t_e2e * 1e3], device=dev, dtype=torch.float64)
    if world > 1:
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    ms_max, e2e_ms_max = float(t[0]), float(t[1])
    if rank != 0:
        return
    value = world * K / (ms_max * 1e-3)
    out = {
        "metric": METRIC, "value": round(value, 4), "unit": "steps/s", "n_gpus": world, "steps": K, "warmup": Wm,
        "ms_per_step": round(ms_max / K, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f16", "data": "synthetic (seeded latents/embeddings, random-init I2VGen-XL UNet 1.42B params)",
        "config": {"workload": f"i2vgen-xl {F}f x 512x512 (latents 1x4x{F}x64x64), 50+50-step DDIM schedules: K/2 inversion steps "
                               "(UNet batch 1) + K/2 PnP edit steps (UNet batch 3, "
                               + ("conv + spatial-attn injection every step" if F == 16 else "conv + spatial + temporal injection every step")
                               + "), cfg 9.0" + ("" if F == 16 else " — BASELINE configs[4], the gradio long-video pattern"),
                   "clips_per_gpu": 1, "pnp": pnp, "parallelism": f"clip-per-gpu x{world} (weights: one NCCL broadcast)",
                   "peak_memory_gb": round(peak_mem_gb, 2),
                   "parity": "DDIM / CFG step bit-exact vs the oracle; kernels vs fp32 restatements at rtol 1e-3 + 1e-3..2e-3 x max|ref| "
                             "(one fp16 rounding is 4.9e-4 relative; north_star's literal atol 1e-4 is below fp16 resolution for |x| > 0.2); "
                             "full-width (1.42 B params) hooked UNet steps as close to the fp32 oracle as torch fp16 is (x3) — tests/",
                   "l2": "per-step working set (2.84 GB fp16 weights + activations) >> 126 MB L2; no explicit flush",
                   "ms_per_inversion_step": round(ms_inv, 3), "ms_per_edit_step": round(ms_edit, 3),
                   "effective_tflops_reference_flops": round((k_inv * TFLOP_INV + k_edit * TFLOP_EDIT) * (F / 16) / (ms_max * 1e-3), 1),
                   "outputs_finite": finite, "model_build_s": round(build_s, 1)},
        "e2e": {"value": round(world * K / (e2e_ms_max * 1e-3), 4), "unit": "steps/s",
                "h2d_bytes_per_step": int(h2d_total // K), "d2h_bytes_per_step": int(d2h_total // K),
                "how": "invert_step / edit_step of anyv2v_b200.pipeline with a pinned-host latent store: conditioning + initial "
                       "latents H2D at the start, per edit step the source latent H2D, per step the new latent D2H (twice: into "
                       "the store and as the step result)"},
        "gpu_launches": int(launches), "cuda_graphs": bool(graphs),
        "clocks": clocks,
        "roofline": roof,
        "roofline_more": roof_more,
        "sub_records": sub,
        "weights_broadcast": getattr(unet, "_broadcast_stats", None),
    }
    if F != 16:
        out["metric"] = METRIC.replace("16f", f"{F}f")
    if not args.no_cpu_baseline and world >= 1:
        out["cpu_baseline"] = cpu_baseline(budget_s=args.cpu_budget)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last_outputs)
    print(json.dumps(out), flush=True)


DUMP_BYTES = 60 * 2 ** 20


def dump_outputs(out_dir, arrays):
    """Write each array as out_dir/<name>.npy in float32, DUMP_BYTES at most in all.  An array larger than its share is replaced by
    a seeded sample of its elements, the same positions in every run, so that two builds can be compared output for output."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // 4 // max(len(arrays), 1)
    for name, t in arrays.items():
        if t.numel() > share:
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:share].sort().values
            t = t.reshape(-1)[idx]
        np.save(os.path.join(out_dir, f"{name}.npy"), t.numpy().astype(np.float32))


def attention_roofline(ops, dev):
    """The injected spatial self-attention at the finest level (N = 4096 tokens, 5 heads, 16 source frames, probabilities
    shared by the 3 branches): algorithmic FLOPs = QK^T once + PV for 3 branches = 2*T*L*64*(1+3) per head-batch."""
    peaks = measured_peaks()
    heads, seq, batch = 5, 4096, F
    C = heads * 64
    rows = batch * seq
    qk = torch.randn(rows, 2 * C, device=dev).half()
    v = torch.randn(3 * rows, C, device=dev).half()
    out = torch.empty(3 * rows, C, device=dev, dtype=torch.float16)
    fn = lambda: ops.attention(qk[:, :C], qk[:, C:], v, heads, seq, batch, out, n_v=3, v_branch_stride=rows * C, o_branch_stride=rows * C)
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    iters = 20
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    dur = e0.elapsed_time(e1) / iters * 1e-3
    flops = 2.0 * batch * heads * seq * seq * 64 * (1 + 3)
    achieved = flops / dur / 1e12
    return {"kernel": "attn_pnp_kernel<3> (spatial PnP self-attention, up_blocks[3] site: 16 src frames x 5 heads x 4096 tokens, shared P)",
            "bound": "tensor", "achieved": round(achieved, 1), "peak": peaks["tflops_burst"], "unit": "TFLOP/s",
            "frac": round(achieved / peaks["tflops_burst"], 4),
            # dram__bytes_read.sum + dram__bytes_write.sum per launch of this geometry, read at run time from the committed
            # `ncu --set full` capture (null when the file is absent); algorithmic minimum 0.34 GB (q, k + 3 v + 3 o)
            **ncu_traffic(("r02_attn3.ncu.csv", "r01_prof_attn3_v9.ncu.csv"), "attn_pnp_kernel"),
            "peak_source": peaks["source"] + ", burst (kernel timed alone, back-to-back launches, q/k/v 0.25 GB > L2)",
            "us_per_launch": round(dur * 1e6, 1),
            "algorithmic_flops_per_launch": flops}


def ncu_traffic(csv_names, kernel_substr):
    """{"traffic": dram__bytes_read.sum + dram__bytes_write.sum of `kernel_substr`'s launch in the first committed ncu summary of
    `csv_names` under profiles/ (`metric,unit,value` rows written by tools/ncu_extract.py from an `ncu --set full` report),
    "traffic_unit": where it came from}; traffic = None when no capture is committed — never a constant typed into this file."""
    import csv
    scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    for name in csv_names:
        path = os.path.join(ROOT, "profiles", name)
        if not os.path.exists(path):
            continue
        try:
            with open(path, newline="") as fh:
                rows = {r[0]: r for r in csv.reader(fh) if len(r) >= 3}
            if kernel_substr not in rows["Kernel Name"][2]:
                continue
            tot = sum(float(rows[m][2].replace(",", "")) * scale[rows[m][1]] for m in ("dram__bytes_read.sum", "dram__bytes_write.sum"))
            return {"traffic": tot, "traffic_unit": f"bytes/launch (ncu dram__bytes_read.sum + dram__bytes_write.sum, profiles/{name})"}
        except (KeyError, ValueError, IndexError, OSError):
            continue
    return {"traffic": None, "traffic_unit": "no committed ncu capture found under profiles/"}


def _time_us(fn, iters=20, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1e3


def temporal_attention_roofline(ops, dev):
    """The temporal self-attention of a PnP-injected step at the finest level (pnp_utils.py:247-334; 3 branches x 16 frames x
    4096 pixels, C = 320, 5 heads): ONE kernel, Q/K/V projection + SDPA, Q and K projected from the source clip.  HBM-bound:
    algorithmic bytes = the tokens read once + the output written once (the 0.6 MB of weights are L2-resident)."""
    peaks = measured_peaks()
    heads, frames, hw, clips = 5, 16, 4096, 3
    C = heads * 64
    rows = clips * frames * hw
    x = torch.randn(rows, C, device=dev).half()
    w = (torch.randn(3 * C, C, device=dev) / C ** 0.5).half()
    out = torch.empty(rows, C, device=dev, dtype=torch.float16)
    us = _time_us(lambda: ops.temporal_attention_fused(x, w, heads, frames, hw, clips, out, n_v=3))
    nbytes = 2.0 * rows * C * 2
    gbs = nbytes / us / 1e3
    return {"kernel": "tattn_fused2_kernel, injected (temporal PnP self-attention, up_blocks[3] site: [src|uncond|cond] x 16 f x 4096 px, C 320)",
            "bound": "hbm", "achieved": round(gbs, 1), "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": round(gbs / peaks["hbm_gbs"], 4),
            **ncu_traffic(("r02_tattn_fused.ncu.csv",), "tattn_fused"), "us_per_launch": round(us, 1),
            "algorithmic_bytes_per_launch": nbytes, "peak_source": peaks["source"],
            "note": "projection FLOPs 2*rows*320*960 + 3x re-projected q,k (injected variant) make this kernel L2->SM-fabric bound, "
                    "not HBM-bound, today: see DESIGN.md"}


def groupnorm_roofline(ops, dev):
    """GroupNorm+SiLU of a clip-level norm at the finest level (TemporalConvLayer, [3, 65536, 320]): 4 B per element."""
    peaks = measured_peaks()
    n, rows, C = 3, 65536, 320
    x = torch.randn(n, rows, C, device=dev).half()
    g, b = torch.randn(C, device=dev).half(), torch.randn(C, device=dev).half()
    o = torch.empty_like(x)
    us = _time_us(lambda: ops.groupnorm(x, g, b, 32, 1e-5, True, out=o))
    nbytes = 4.0 * n * rows * C
    gbs = nbytes / us / 1e3
    return {"kernel": "gn_persistent_kernel (GroupNorm+SiLU [3, 65536, 320], TemporalConvLayer norms of the 64x64 level)", "bound": "hbm",
            "achieved": round(gbs, 1), "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": round(gbs / peaks["hbm_gbs"], 4),
            **ncu_traffic(("r02_groupnorm.ncu.csv",), "gn_persistent_kernel"), "us_per_launch": round(us, 1),
            "algorithmic_bytes_per_launch": nbytes, "peak_source": peaks["source"]}


def gemm_rooflines(ops, dev):
    """The GEMM kernel is the dominant kernel of the step by time (~60 %): two of its heaviest shapes, timed live.  (1) the
    attention-block projection at the finest level, K = 320 (to_q|to_k|to_v of 3 x 16 frames x 4096 tokens: 196608 x 960 x 320), on
    the machine's ridge: reported against BOTH bounds; (2) the GEGLU feed-forward GEMM of the same level (196608 x 2560 x 320,
    h * gelu(gate) fused, 1280 output columns)."""
    peaks = measured_peaks()
    out = []
    M, K = 196608, 320
    a = torch.randn(M, K, device=dev).half()
    for name, N, geglu, csv_name in (("linear 196608x960x320 (+bias; q|k|v projection of the 64x64 level)", 960, False, "r02_gemm_lin960.ncu.csv"),
                                     ("linear+GEGLU 196608x2560x320 (feed-forward of the 64x64 level, 1280 output columns)", 2560, True, "r02_gemm_geglu.ncu.csv")):
        w = (torch.randn(N, K, device=dev) / 18).half()
        b = torch.randn(N, device=dev).half()
        if geglu:
            w, b = ops.geglu_pack(w, b)
        o = torch.empty(M, N // 2 if geglu else N, device=dev, dtype=torch.float16)
        us = _time_us(lambda: ops.linear(a, w, bias=b, geglu=geglu, out=o))
        flops = 2.0 * M * N * K
        nbytes = 2.0 * (M * K + N * K + o.numel())
        tf, gbs = flops / us / 1e6, nbytes / us / 1e3
        t_tensor, t_hbm = flops / (peaks["tflops_sustained"] * 1e6), nbytes / (peaks["hbm_gbs"] * 1e3)
        bound = "tensor" if t_tensor >= t_hbm else "hbm"
        out.append({"kernel": f"gemm_tcgen05_kernel ({name})", "bound": bound,
                    "achieved": round(tf if bound == "tensor" else gbs, 1),
                    "peak": peaks["tflops_sustained"] if bound == "tensor" else peaks["hbm_gbs"],
                    "unit": "TFLOP/s" if bound == "tensor" else "GB/s",
                    "frac": round(max(t_tensor, t_hbm) / us, 4), **ncu_traffic((csv_name,), "gemm_tcgen05_kernel"),
                    "us_per_launch": round(us, 1), "algorithmic_flops_per_launch": flops, "algorithmic_bytes_per_launch": nbytes,
                    "tensor_bound_us": round(t_tensor, 1), "hbm_bound_us": round(t_hbm, 1),
                    "peak_source": peaks["source"] + ", sustained (the kernel runs inside a long power-capped step)"})
        del w, b, o
    return out


def config3_record(pipe, edit_sched, cond_dev, dev, ms_inv, init_pnp):
    """BASELINE.json configs[2] (template defaults' siblings: pnp_f_t 0.8 -> conv injection on edit steps 0-39, pnp_spatial_attn_t =
    pnp_temp_attn_t 0.5 -> both attention injections on steps 0-24; reference schedule arithmetic run_group_pnp_edit.py:35-48).
    The 50 edit steps fall into three classes, each with its own captured CUDA graph: all three hooks fire (25 steps), conv only
    (15), nothing fires = the source branch is dead and not run (10).  Per class: 1 eager + 1 capture step, then 3 timed replays."""
    from types import SimpleNamespace
    from anyv2v_b200.latent_store import LatentStore
    init_pnp(pipe, edit_sched, SimpleNamespace(n_steps=N_SCHEDULE, **PNP_CONFIG3))
    store = LatentStore(None, write_files=False)
    g = torch.Generator().manual_seed(777)
    for t in edit_sched.timesteps.tolist():
        store.put(int(t), torch.randn(1, 4, F, H, W, generator=g).half().to(dev))
    st = pipe.prepare_edit(cond_dev["video_latents"].clone(), cond_dev["edit_prompt"], cond_dev["neg_prompt"], cond_dev["inv_prompt"],
                           cond_dev["edit_image_emb"], cond_dev["edit_image_latents"], cond_dev["src_image_emb"],
                           cond_dev["src_image_latents"], 8, N_SCHEDULE, GUIDANCE, 0, None, store, True)
    classes = (("conv+spatial+temporal", 0, 25), ("conv_only", 25, 15), ("dead_source", 40, 10))
    ms = {}
    for name, i0, _count in classes:
        for i in range(i0, i0 + 2):
            pipe.edit_step(st, i)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(i0 + 2, i0 + 5):
            pipe.edit_step(st, i)
        e1.record()
        torch.cuda.synchronize()
        ms[name] = e0.elapsed_time(e1) / 3
    job_ms = 50 * ms_inv + sum(cnt * ms[name] for name, _i0, cnt in classes)
    return {"workload": "BASELINE configs[2]: 16f x 512^2, 50 inversion + 50 PnP edit steps, pnp_f_t 0.8 / pnp_spatial_attn_t 0.5 / "
                        "pnp_temp_attn_t 0.5 (conv injection on 40 steps, spatial + temporal attention injection on 25)",
            "pnp": PNP_CONFIG3, "ms_per_edit_step": {k: round(v, 3) for k, v in ms.items()},
            "edit_steps_per_class": {name: cnt for name, _i0, cnt in classes}, "ms_per_inversion_step": round(ms_inv, 3),
            "value": round(100.0 / (job_ms * 1e-3), 4), "unit": "steps/s",
            "how": "100 / (50 x inversion step + 25 x all-hooks step + 15 x conv-only step + 10 x dead-source step); per-class times are "
                   "CUDA-event means of 3 graph replays in this run",
            "outputs_finite": bool(torch.isfinite(st.latents).all())}


# =============================================================================================== CPU reference arm
_CPU_NET = None


def _cpu_net():
    """the full-size fp32 oracle UNet (1.42 B parameters), built once per process"""
    global _CPU_NET
    if _CPU_NET is None:
        from oracle import unet_ref
        _CPU_NET = unet_ref.seeded_unet(unet_ref.I2VGEN_XL_CONFIG, seed=8888, dtype=torch.float32, device="cpu")
    return _CPU_NET


def _cpu_step_times(frames: int, n_inv: int, n_edit: int, pnp=None):
    """Times n_inv inversion steps and n_edit PnP-edit steps of the oracle (reference CPU port) at `frames` frames."""
    from types import SimpleNamespace

    from oracle import loops_ref, pnp_hooks_ref as hooks, schedulers_ref as sref
    net = _cpu_net()
    ns = loops_ref.synthetic_inputs(frames, H, W, cross_dim=1024, seed=8888, dtype=torch.float32)
    pipe = SimpleNamespace(unet=net)
    s = sref.DDIMScheduler()
    s.set_timesteps(N_SCHEDULE)
    inv = sref.DDIMInverseScheduler()
    inv.set_timesteps(N_SCHEDULE)
    prompts, img_lat, img_emb, fps3 = loops_ref.edit_conditioning(ns)
    lat = ns.video_latents
    t_inv, t_edit = [], []
    with torch.no_grad():
        hooks.init_pnp(pipe, s, N_SCHEDULE, 0.0, 0.0, 0.0)  # the inversion process registers no hooks
        hooks.register_time(pipe, -1)
        for i in range(n_inv):
            t = int(inv.timesteps[i])
            t0 = time.perf_counter()
            v = net(lat, torch.tensor(t), ns.fps, ns.src_image_latents, ns.src_image_emb, ns.inv_prompt)[0]
            lat, _ = inv.step(v, t, lat)
            t_inv.append(time.perf_counter() - t0)
        hooks.init_pnp(pipe, s, N_SCHEDULE, **(pnp or PNP))  # the reference registers the hooks in the edit process only
        x = ns.video_latents.clone()
        for i in range(n_edit):
            t = int(s.timesteps[i])
            t0 = time.perf_counter()
            hooks.register_time(pipe, t)
            v = net(torch.cat([lat, x, x]), torch.tensor(t), fps3, img_lat, img_emb, prompts)[0]
            x, _ = s.step(sref.cfg_combine(v[1:2], v[2:3], GUIDANCE), t, x)
            t_edit.append(time.perf_counter() - t0)
    return t_inv, t_edit


def _fit_frames(points, target_frames):
    """least-squares line t(f) = a + b f through [(frames, seconds)] -> (t(target_frames), a, b, max relative residual).
    The oracle's cost is linear in the frame count apart from the per-call overheads (a) and the temporal attention (F^2, 0.1 %
    of the FLOPs at F = 16): the residual says how well that holds on this host."""
    n = len(points)
    if n == 1:
        f, t = points[0]
        return t * target_frames / f, 0.0, t / f, None
    sx = sum(f for f, _ in points)
    sy = sum(t for _, t in points)
    sxx = sum(f * f for f, _ in points)
    sxy = sum(f * t for f, t in points)
    b = (n * sxy - sx * sy) / (n * sxx - sx * sx)
    a = (sy - b * sx) / n
    resid = max(abs(a + b * f - t) / t for f, t in points)
    return a + b * target_frames, a, b, resid


def _cpu_measure(budget_s: float, reps_cap: int = 1):
    """(inversion step, edit step) of the full-size oracle at 1, 2 and 4 of the F frames — as many of the three as fit the
    budget — each fitted to a line in the frame count and evaluated at F frames."""
    t_begin = time.perf_counter()
    pts_inv, pts_edit, note = [], [], []
    for frames in (1, 2, 4):
        if pts_inv:
            per_frame = (pts_inv[-1][1] + pts_edit[-1][1]) / pts_inv[-1][0]
            if time.perf_counter() - t_begin + per_frame * frames * 1.1 > budget_s:
                break
        reps = 1
        if pts_inv and reps_cap > 1:
            reps = int(max(1, min(reps_cap, (budget_s - (time.perf_counter() - t_begin)) / (per_frame * frames * 3.0))))
        ti, te = _cpu_step_times(frames, reps, reps)
        pts_inv.append((frames, sum(ti) / len(ti)))
        pts_edit.append((frames, sum(te) / len(te)))
        note.append(f"{frames}f: inv {pts_inv[-1][1]:.2f}s edit {pts_edit[-1][1]:.2f}s (x{reps})")
    inv_s, a_i, b_i, r_i = _fit_frames(pts_inv, F)
    edit_s, a_e, b_e, r_e = _fit_frames(pts_edit, F)
    resid = None if r_i is None else max(r_i, r_e)
    how = (f"full-size fp32 oracle (CPU port of the reference path), 512x512, timed at {', '.join(note)}; per-step time fitted as "
           f"a + b*frames (inv: a={a_i:.2f}s b={b_i:.2f}s/frame; edit: a={a_e:.2f}s b={b_e:.2f}s/frame"
           + (f"; max relative residual of the fit {resid:.1%}" if resid is not None else "; single point, proportional scaling")
           + f") and evaluated at {F} frames: inversion step {inv_s:.1f}s, PnP edit step {edit_s:.1f}s")
    return inv_s, edit_s, how, resid


def cpu_baseline(budget_s: float = 40.0):
    """Oracle (= CPU port of the reference path: restated diffusers UNet + reference hook/loop arithmetic) on the host cores,
    on a bounded sample: the full-size UNet at 512x512 with 1, 2 and 4 of the frames, 1 inversion + 1 edit step each, fitted
    in the frame count (see _cpu_measure) — not a plain x16."""
    cores = _calibrated_threads(_usable_cores())
    inv_s, edit_s, how, resid = _cpu_measure(budget_s)
    return {"value": round(2.0 / (inv_s + edit_s), 6), "unit": "steps/s", "cores": cores, "kind": "port", "sample": how,
            "fit_max_rel_residual": resid, "cpu": _cpu_name()}


def _usable_cores() -> int:
    """Host threads the CPU arms may really use: the affinity mask capped by the cgroup CPU quota (a 128-CPU box with a
    16-CPU quota thrashes when 128 threads are started — measured 30x slower than 8 threads on an 8-CPU box)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except (AttributeError, OSError):
        pass
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, -(-int(txt[0]) // int(txt[1]))))
            else:
                quota = int(txt[0])
                period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                if quota > 0:
                    n = min(n, max(1, -(-quota // period)))
            break
        except (OSError, ValueError, IndexError):
            continue
    return n


def _calibrated_threads(cores: int) -> int:
    """Pick the torch thread count that is actually fastest on this host for the CPU arm's dominant op (a 3x3 fp32
    convolution at the sample's size): more threads than the host can schedule only adds contention."""
    import torch.nn.functional as F
    x = torch.randn(2, 320, 64, 64)
    w = torch.randn(320, 320, 3, 3)
    best, best_t = cores, float("inf")
    cand = sorted({c for c in (cores, cores // 2, cores // 4, 32, 16, 8) if 1 <= c <= cores}, reverse=True)
    for c in cand:
        torch.set_num_threads(c)
        F.conv2d(x, w, padding=1)
        t0 = time.perf_counter()
        for _ in range(3):
            F.conv2d(x, w, padding=1)
        dt = time.perf_counter() - t0
        if dt < best_t * 0.95:
            best, best_t = c, dt
    torch.set_num_threads(best)
    return best


def _cpu_name():
    try:
        with open("/proc/cpuinfo") as fh:
            for l in fh:
                if l.startswith("model name"):
                    return l.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def run_reference(args):
    """Reference arm: the reference's own CPU implementation of the path.  The reference cannot be installed (its UNet
    lives in diffusers==0.26.3, which is neither in /root/reference nor in the wheelhouse), so this times the oracle
    port with all host threads.  Each step is a bounded sample: the full-size model at 1, 2 and 4 of the frames, fitted in the
    frame count and evaluated at the full clip (the fit's residual is reported)."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    cores = _calibrated_threads(_usable_cores())
    K, Wm = args.steps, args.warmup
    k_inv, k_edit = (K + 1) // 2, K // 2
    pnp = PNP_LONG if F > 16 else PNP
    inv_s, edit_s, how, resid = _cpu_measure(args.ref_budget, reps_cap=3)
    total = k_inv * inv_s + k_edit * edit_s
    value = K / total  # the CPU arm does not scale with --gpus: one host, one clip at a time
    metric = METRIC if F == 16 else METRIC.replace("16f", f"{F}f")
    out = {"impl": "reference", "metric": metric, "value": round(value, 6), "unit": "steps/s", "n_gpus": args.gpus, "steps": K,
           "warmup": Wm, "ms_per_step": round(total / K * 1e3, 1), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "f32", "data": "synthetic (seeded latents/embeddings, random-init I2VGen-XL UNet 1.42B params)",
           "config": {"workload": f"same as the GPU arm ({F}f x 512x512, K/2 inversion + K/2 PnP edit steps, injection every step)", "pnp": pnp,
                      "note": "reference cannot be pip-installed offline (needs diffusers==0.26.3); oracle CPU port timed instead"},
           "cpu_baseline": {"value": round(value, 6), "unit": "steps/s", "cores": cores, "kind": "port", "cpu": _cpu_name(),
                            "sample": how + f"; K={K} steps extrapolated from those two per-step times", "fit_max_rel_residual": resid},
           "e2e": {"value": round(value, 6), "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--impl", type=str, default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--frames", type=int, default=16, help="frames per clip: 16 (BASELINE configs[1], default) or 128 (configs[4])")
    ap.add_argument("--cpu-budget", type=float, default=40.0)
    ap.add_argument("--ref-budget", type=float, default=150.0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the latents the last timed inversion step and edit step returned (rank 0) "
                         "as DIR/inversion_latents.npy and DIR/edit_latents.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl ours: the reference arm only times the oracle")
    global F
    F = args.frames
    if args.warmup < 4:
        args.warmup = 4  # 2 + 2: per phase one eager pass and one CUDA-graph capture before the timed region
    if args.impl == "reference":
        run_reference(args)
    else:
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device — the product path has no CPU fallback (use --impl reference for the CPU arm)")
        run_ours(args)
        if torch.distributed.is_initialized():
            torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()

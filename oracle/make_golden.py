"""ORACLE (test infrastructure): pin the restatement against what /root/reference itself holds, and freeze golden
vectors into tests/golden/.  Runs ONLY in the build container (needs /root/reference); the committed fixtures then
travel to the GPU box.  Usage:  python -m oracle.make_golden

What is pinned here (the reference has no tests; diffusers is absent — see oracle/__init__.py):
  1. the UNMODIFIED reference hooks  i2vgen-xl/pnp_utils.py  executed on the oracle UNet (through diffusers_shim)
     == the oracle's restated hooks (oracle/pnp_hooks_ref.py), bit for bit, at an injected step, a non-injected
     step and the t == 1000 special case;
  2. the reference's vendored scheduler  consisti2v/ddim_inverse_scheduler.py  == oracle/schedulers_ref.py
     (alphas_cumprod, timesteps, inverse step), bit for bit in fp32;
  3. golden outputs of (1) and (2) on seeded inputs -> tests/golden/*.pt
"""
from __future__ import annotations

import os
import shutil
from types import SimpleNamespace

import torch

from . import diffusers_shim, loops_ref, pnp_hooks_ref, schedulers_ref, unet_ref

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
TINY = dict(F=4, h=16, w=16)


def tiny_case(seed=8888):
    ns = loops_ref.synthetic_inputs(TINY["F"], TINY["h"], TINY["w"], cross_dim=unet_ref.TINY_CONFIG["cross_attention_dim"], seed=seed)
    prompts, img_lat, img_emb, fps = loops_ref.edit_conditioning(ns)
    g = torch.Generator().manual_seed(seed + 7)
    x3 = torch.randn(3, 4, TINY["F"], TINY["h"], TINY["w"], generator=g)
    return x3, prompts, img_lat, img_emb, fps


def run_hooks(hooks_mod, t: int, schedule):
    pipe = SimpleNamespace(unet=unet_ref.seeded_unet(unet_ref.TINY_CONFIG, seed=8888))
    hooks_mod.register_conv_injection(pipe, schedule)
    hooks_mod.register_spatial_attention_pnp(pipe, schedule)
    hooks_mod.register_temp_attention_pnp(pipe, schedule)
    hooks_mod.register_time(pipe, t)
    x3, prompts, img_lat, img_emb, fps = tiny_case()
    with torch.no_grad():
        return pipe.unet(x3, torch.tensor(t), fps, img_lat, img_emb, prompts)[0]


def main():
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(max(1, (os.cpu_count() or 2) // 2))
    ref_hooks = diffusers_shim.load_reference_module("i2vgen-xl/pnp_utils.py", "ref_pnp_utils")
    ref_sched_mod = diffusers_shim.load_reference_module("consisti2v/ddim_inverse_scheduler.py", "ref_inv_sched")

    # ---- 1. hooks: reference file vs restatement
    sched = schedulers_ref.DDIMScheduler()
    sched.set_timesteps(10)
    schedule = sched.timesteps[:5]  # [901, 801, 701, 601, 501]
    golden = {"schedule": schedule.clone(), "tiny": dict(TINY)}
    for name, t in (("injected", 901), ("not_injected", 101), ("t1000", 1000)):
        a = run_hooks(ref_hooks, t, schedule)
        b = run_hooks(pnp_hooks_ref, t, schedule)
        assert torch.equal(a, b), f"restated hooks differ from the reference at t={t}: {(a - b).abs().max()}"
        golden[name] = a.clone()
        print(f"hooks {name:13s} t={t}: reference == restatement (bit-exact), |out| mean {a.abs().mean():.4f}")
    # empty schedule == unpatched model (Appendix C.5)
    plain = SimpleNamespace(unet=unet_ref.seeded_unet(unet_ref.TINY_CONFIG, seed=8888))
    x3, prompts, img_lat, img_emb, fps = tiny_case()
    with torch.no_grad():
        base = plain.unet(x3, torch.tensor(901), fps, img_lat, img_emb, prompts)[0]
    none = run_hooks(ref_hooks, 901, [])
    assert torch.equal(base, none), "empty injection schedule must equal the unpatched model"
    assert not torch.equal(base, golden["injected"])
    golden["unpatched"] = base.clone()
    torch.save(golden, os.path.join(OUT, "tiny_unet_pnp.pt"))

    # ---- 2. scheduler: vendored reference class vs restatement
    ref_s = ref_sched_mod.DDIMInverseScheduler(**schedulers_ref.CONFIG)
    ours = schedulers_ref.DDIMInverseScheduler()
    assert torch.equal(ref_s.alphas_cumprod, ours.alphas_cumprod)
    kat = {"alphas_idx": torch.tensor([0, 1, 21, 41, 481, 501, 961, 981, 999])}
    kat["alphas"] = ours.alphas_cumprod[kat["alphas_idx"]].clone()
    g = torch.Generator().manual_seed(123)
    x = torch.randn(2, 4, 8, 8, generator=g)
    v = torch.randn(2, 4, 8, 8, generator=g)
    kat["x"], kat["v"] = x, v
    for n in (10, 50, 500):
        ref_s.set_timesteps(n)
        ours.set_timesteps(n)
        assert torch.equal(ref_s.timesteps, ours.timesteps)
        kat[f"timesteps_{n}"] = ours.timesteps.clone()
        for t in (int(ours.timesteps[0]), int(ours.timesteps[n // 2]), int(ours.timesteps[-1])):
            a = ref_s.step(v, t, x).prev_sample
            b, _ = ours.step(v, t, x)
            assert torch.equal(a, b), f"inverse step differs at n={n} t={t}"
            kat[f"inv_step_{n}_{t}"] = a.clone()
    torch.save(kat, os.path.join(OUT, "scheduler_kat.pt"))
    print("scheduler: vendored reference class == restatement (alphas, timesteps, inverse step) — bit-exact")

    # ---- the reference's config templates, verbatim, for the config API test
    for rel in ("group_pnp_edit/template.yaml", "group_pnp_edit/group_config.json", "group_ddim_inversion/template.yaml"):
        dst = os.path.join(OUT, "reference_configs", rel)
        os.makedirs(os.path.dirname(dst), exist_ok=True)
        shutil.copyfile(os.path.join(diffusers_shim.REF_ROOT, "i2vgen-xl", "configs", rel), dst)
    for f in sorted(os.listdir(OUT)):
        print(f"  tests/golden/{f}: {os.path.getsize(os.path.join(OUT, f))} bytes")


if __name__ == "__main__":
    main()

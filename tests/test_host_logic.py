"""CPU tests of the host-side logic: C-ABI exports, config API, schedules, hook registration semantics, scheduler
host side vs the oracle, latent files, and the world_size-2 (gloo) weight broadcast / clip sharding."""
import ctypes
import json
import os
import re
import subprocess
import sys
from types import SimpleNamespace

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_cabi_library_exports_every_declared_symbol():
    import __graft_entry__ as g
    g.build()
    from anyv2v_b200 import _lib
    lib = _lib.lib()
    header = open(os.path.join(ROOT, "include", "anyv2v_b200.h")).read()
    declared = set(re.findall(r"\b(av2v_[a-z0-9_]+)\s*\(", header))
    assert declared == set(_lib.EXPORTS), (declared ^ set(_lib.EXPORTS))
    for name in declared:
        assert hasattr(lib, name), f"{name} is declared in include/anyv2v_b200.h but not exported"
    assert lib.av2v_abi_version() == 1
    assert lib.av2v_groupnorm_workspace_floats(2, 320) == 2 * 512 * 64 * 2
    # argument validation happens before any CUDA call, so it can be exercised without a GPU
    a = _lib.GemmArgs()
    assert lib.av2v_gemm_f16(ctypes.byref(a), None) == _lib.AV2V_EINVAL
    assert b"null" in lib.av2v_last_error()
    assert lib.av2v_ddim_step_cfg_f16(None, None) == _lib.AV2V_EINVAL


def test_ops_refuse_cpu_tensors_loudly():
    from anyv2v_b200 import ops
    from anyv2v_b200._lib import Av2vError
    with pytest.raises(Av2vError, match="no CPU fallback"):
        ops.linear(torch.zeros(8, 8, dtype=torch.float16), torch.zeros(8, 8, dtype=torch.float16))
    with pytest.raises(Av2vError):
        ops.groupnorm(torch.zeros(1, 4, 32, dtype=torch.float16), torch.ones(32).half(), torch.zeros(32).half(), 32, 1e-5, True)


# the reference's own i2vgen-xl/configs templates (and group_pnp_edit's group_config.json), stored verbatim (oracle/make_golden.py)
REF_CFG = os.path.join(ROOT, "tests", "golden", "reference_configs")


def test_config_api_on_the_reference_templates():
    from anyv2v_b200.config import OmegaConf
    t = OmegaConf.load(f"{REF_CFG}/group_pnp_edit/template.yaml")
    entry = json.load(open(f"{REF_CFG}/group_pnp_edit/group_config.json"))[0]
    c = OmegaConf.merge(t, OmegaConf.create(entry))
    assert c.pnp_f_t == 1.0 and c.ddim_init_latents_t_idx == 0 and c.n_steps == 50 and c.cfg == 9.0
    assert c.output_dir == "../Results/Prompt-Based-Editing/i2vgen-xl/" + entry["video_name"] + "/" + entry["edited_video_name"] + "/"
    assert c.ddim_latents_path == "../inversions/i2vgen-xl/" + entry["video_name"] + "/ddim_latents"
    assert t.pnp_f_t == 0.2  # merge does not mutate the template
    inv = OmegaConf.load(f"{REF_CFG}/group_ddim_inversion/template.yaml")
    c2 = OmegaConf.merge(inv, OmegaConf.create({"video_name": "clip"}))
    assert c2.inverse_config.output_dir == "../inversions/i2vgen-xl/clip/ddim_latents"
    assert c2.inverse_config.image_size == [512, 512] and c2.recon_config.ddim_latents_path == c2.inverse_config.output_dir


def test_config_merge_interpolation_and_assignment(tmp_path):
    from anyv2v_b200.config import OmegaConf
    p = tmp_path / "t.yaml"
    p.write_text("a: 1\nname: ReplaceMe\nout: \"${root}/${name}\"\nroot: /r\nsub:\n  size: ${dims}\n  deep: \"${sub.k}\"\n  k: 3\ndims: [4, 5]\n")
    t = OmegaConf.load(str(p))
    c = OmegaConf.merge(t, OmegaConf.create({"name": "clip", "sub": {"k": 7}}))
    assert c.out == "/r/clip" and c.sub.size == [4, 5] and c.sub.deep == 7 and c["a"] == 1
    c.extra = "x"
    assert c.extra == "x" and "extra" in c and "name: clip" in OmegaConf.to_yaml(c)
    with pytest.raises(AttributeError):
        _ = c.missing


def test_pnp_schedules_match_reference_truncation():
    from anyv2v_b200.run_group_pnp_edit import config_suffix, pnp_schedules
    from anyv2v_b200.schedulers import DDIMScheduler
    s = DDIMScheduler()
    s.set_timesteps(50)
    cfg = SimpleNamespace(n_steps=50, pnp_f_t=0.8, pnp_spatial_attn_t=0.5, pnp_temp_attn_t=-1.0, ddim_init_latents_t_idx=0, cfg=9.0)
    f, sp, tm = pnp_schedules(s, cfg)
    assert f.tolist() == list(range(981, 981 - 800, -20)) and len(sp) == 25 and len(tm) == 0
    cfg.pnp_f_t = 0.58
    assert len(pnp_schedules(s, cfg)[0]) == 28  # int(50*0.58) float truncation, run_group_pnp_edit.py:36
    assert config_suffix(cfg) == "ddim_init_latents_t_idx_0_nsteps_50_cfg_9.0_pnpf0.58_pnps0.5_pnpt-1.0"


def test_scheduler_host_side_matches_oracle():
    from anyv2v_b200 import schedulers
    from oracle import schedulers_ref
    for ours_cls, ref_cls in ((schedulers.DDIMScheduler, schedulers_ref.DDIMScheduler),
                              (schedulers.DDIMInverseScheduler, schedulers_ref.DDIMInverseScheduler)):
        ours, ref = ours_cls(), ref_cls()
        assert torch.equal(ours.alphas_cumprod, ref.alphas_cumprod)
        for n in (10, 50, 500):
            ours.set_timesteps(n)
            ref.set_timesteps(n)
            assert ours.timesteps.tolist() == ref.timesteps.tolist()
            for t in ours.timesteps.tolist()[:: max(1, n // 7)]:
                assert ours.coefficients(t) == ref.coefficients(t)
    with pytest.raises(ValueError):
        schedulers.DDIMScheduler().set_timesteps(2000)
    with pytest.raises(ValueError):
        schedulers.DDIMScheduler(prediction_type="epsilon")


def _tiny_pipe():
    from anyv2v_b200.unet_i2vgen_xl import I2VGenXLUNet
    from oracle.unet_ref import TINY_CONFIG
    return SimpleNamespace(unet=I2VGenXLUNet(**TINY_CONFIG))


def test_hook_registration_semantics():
    """Side effects of the four entry points equal the reference's (pnp_utils.py:19-28, 130-132, 235-242, 340-346)."""
    from anyv2v_b200 import pnp_utils as h
    pipe = _tiny_pipe()
    sched = torch.tensor([901, 801, 701])
    h.register_conv_injection(pipe, sched)
    h.register_spatial_attention_pnp(pipe, sched)
    h.register_temp_attention_pnp(pipe, [])
    res = pipe.unet.up_blocks[1].resnets[1]
    assert "forward" in res.__dict__ and res.injection_schedule is sched
    assert "forward" not in pipe.unet.up_blocks[1].resnets[0].__dict__
    patched, plain = 0, 0
    for r in (1, 2, 3):
        for b in range(3):
            for stack, cls in ((pipe.unet.up_blocks[r].attentions, h.ModifiedSpaAttnProcessor),
                               (pipe.unet.up_blocks[r].temp_attentions, h.ModifiedTmpAttnProcessor)):
                proc = stack[b].transformer_blocks[0].attn1.processor
                if (r, b) == (1, 0):
                    assert not isinstance(proc, cls)
                    plain += 1
                else:
                    assert isinstance(proc, cls)
                    patched += 1
    assert patched == 16 and plain == 2
    h.register_time(pipe, 801)
    assert res.t == 801
    sp = pipe.unet.up_blocks[3].attentions[2].transformer_blocks[0].attn1.processor
    tp = pipe.unet.up_blocks[3].temp_attentions[2].transformer_blocks[0].attn1.processor
    assert sp.t == 801 and sp.inject_now() and not tp.inject_now()
    # register_time also reaches the un-patched up_blocks[1].*[0] processors, like the reference
    assert pipe.unet.up_blocks[1].attentions[0].transformer_blocks[0].attn1.processor.t == 801
    h.register_time(pipe, 101)
    assert not sp.inject_now()
    h.register_time(pipe, 1000)  # t == 1000 forces injection wherever a schedule object exists, even an empty one
    assert sp.inject_now() and tp.inject_now()      # (`schedule is not None and (t in schedule or t == 1000)`)
    # idempotent re-registration (init_pnp runs once per clip on the same pipe)
    h.register_spatial_attention_pnp(pipe, sched)
    assert isinstance(pipe.unet.up_blocks[3].attentions[2].transformer_blocks[0].attn1.processor, h.ModifiedSpaAttnProcessor)
    assert h.register_temporal_attention_pnp is h.register_temp_attention_pnp


def test_state_dict_names_equal_the_oracle_model():
    from anyv2v_b200.unet_i2vgen_xl import I2VGEN_XL_CONFIG, I2VGenXLUNet
    from oracle import unet_ref
    with torch.device("meta"):
        a = I2VGenXLUNet(**I2VGEN_XL_CONFIG)
        b = unet_ref.I2VGenXLUNet(**unet_ref.I2VGEN_XL_CONFIG)
    sa = {k: tuple(v.shape) for k, v in a.state_dict().items()}
    sb = {k: tuple(v.shape) for k, v in b.state_dict().items()}
    assert sa == sb and len(sa) == 1511
    assert sum(p.numel() for p in a.parameters()) == 1420469224


def test_latent_store_roundtrip_reference_file_format(tmp_path):
    from anyv2v_b200.latent_store import LatentStore, latent_path, load_ddim_latents_at_T, load_ddim_latents_at_t
    d = str(tmp_path / "ddim_latents")
    store = LatentStore(d)
    xs = {t: torch.randn(1, 4, 2, 4, 4).half() for t in (1, 21, 981)}
    for t, x in xs.items():
        store.put(t, x)
    store.flush()
    assert sorted(os.listdir(d)) == ["ddim_latents_1.pt", "ddim_latents_21.pt", "ddim_latents_981.pt"]
    assert torch.equal(torch.load(latent_path(d, 21)), xs[21])  # plain torch.load, as the reference does (utils.py:28)
    assert torch.equal(load_ddim_latents_at_T(d), xs[981]) and torch.equal(load_ddim_latents_at_t(1, d), xs[1])
    fresh = LatentStore(d, write_files=False)
    assert 981 in fresh and torch.equal(fresh.get(981), xs[981])
    with pytest.raises(AssertionError, match="Missing latents"):
        load_ddim_latents_at_t(5, d)


def test_pipeline_input_errors():
    from anyv2v_b200.pipeline import I2VGenXLPipeline, frame_position_latents
    from anyv2v_b200.schedulers import DDIMScheduler
    pipe = I2VGenXLPipeline(_tiny_pipe().unet, DDIMScheduler())
    with pytest.raises(ValueError, match="prompt_embeds"):
        pipe.sample_with_pnp(prompt="a robot", latents=torch.zeros(1, 4, 2, 8, 8))
    x = frame_position_latents(torch.ones(1, 4, 2, 2), 5)
    assert x.shape == (1, 4, 5, 2, 2) and torch.allclose(x[0, 0, :, 0, 0], torch.tensor([1.0, 0.25, 0.5, 0.75, 1.0]))


def test_gloo_world2_weight_broadcast_and_clip_sharding(tmp_path):
    """N>1 host logic on CPU: rank 0's seeded weights reach rank 1 through ONE broadcast of the flat buffer."""
    script = tmp_path / "w.py"
    script.write_text(f"""
import os, sys, torch, hashlib
sys.path.insert(0, {ROOT!r})
from anyv2v_b200 import distributed
from anyv2v_b200.unet_i2vgen_xl import I2VGenXLUNet
from oracle.unet_ref import TINY_CONFIG
rank, local, world = distributed.init_from_env(backend="gloo")
net = distributed.build_unet_replicated(I2VGenXLUNet, TINY_CONFIG, 8888, "cpu", dtype=torch.float32)
h = hashlib.sha256(net._flat_weights.numpy().tobytes()).hexdigest()
sd = net.state_dict()
ok = all(v.data_ptr() >= net._flat_weights.data_ptr() for v in sd.values())
print("RESULT", rank, world, h, ok, distributed.shard_clips(5, rank, world), flush=True)
""")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    import socket
    with socket.socket() as sock:  # a free port: a fixed one can still be held by a killed earlier run
        sock.bind(("127.0.0.1", 0))
        port = sock.getsockname()[1]
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                          "--master-port", str(port), str(script)], capture_output=True, text=True, timeout=300, env=env)
    lines = [l for l in out.stdout.splitlines() if l.startswith("RESULT")]
    assert len(lines) == 2, out.stdout + out.stderr
    r = sorted(l.split(maxsplit=5) for l in lines)
    assert r[0][3] == r[1][3], "weights differ between ranks after the broadcast"
    assert r[0][4] == r[1][4] == "True"
    assert r[0][5] == "[0, 2, 4]" and r[1][5] == "[1, 3]"


def test_ctypes_structs_match_the_c_header_layout(tmp_path):
    """The Python mirror of the argument structs must have the layout a C compiler gives include/anyv2v_b200.h:
    compile a probe with gcc that prints sizeof / offsetof of every field and compare with ctypes."""
    from anyv2v_b200 import _lib
    structs = {"av2v_ddim_args": _lib.DdimArgs, "av2v_groupnorm_args": _lib.GroupNormArgs, "av2v_gemm_args": _lib.GemmArgs,
               "av2v_layernorm_args": _lib.LayerNormArgs, "av2v_attn_args": _lib.AttnArgs,
               "av2v_tattn_fused_args": _lib.TAttnFusedArgs}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "anyv2v_b200.h"', 'int main(void) {']
    for cname, cls in structs.items():
        lines.append(f'  printf("{cname} %zu\\n", sizeof({cname}));')
        for fname, _ in cls._fields_:
            lines.append(f'  printf("{cname}.{fname} %zu\\n", offsetof({cname}, {fname}));')
    lines += ['  return 0;', '}']
    src = tmp_path / "layout_probe.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout_probe"
    subprocess.run(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    out = dict(l.split() for l in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    for cname, cls in structs.items():
        assert int(out[cname]) == ctypes.sizeof(cls), (cname, out[cname], ctypes.sizeof(cls))
        for fname, _ in cls._fields_:
            assert int(out[f"{cname}.{fname}"]) == getattr(cls, fname).offset, (cname, fname)


def test_bench_cpu_arm_thread_budget_respects_the_cgroup_quota(monkeypatch):
    import bench
    n = bench._usable_cores()
    assert 1 <= n <= (os.cpu_count() or 1)
    try:
        assert n <= len(os.sched_getaffinity(0))
    except AttributeError:
        pass


def test_bench_dump_outputs_float32_within_budget_same_sample(tmp_path, monkeypatch):
    """`bench.py --dump-outputs`: float32 .npy files, an array over its share of the byte budget replaced by the same seeded sample
    of its elements in every run."""
    import numpy as np
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 4000)
    g = torch.Generator().manual_seed(3)
    big, small = torch.randn(1, 4, 16, 8, 8, generator=g).half().float(), torch.randn(2, 3, generator=g)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"big": big, "small": small})
    got = {n: np.load(tmp_path / "a" / f"{n}.npy") for n in ("big", "small")}
    assert all(v.dtype == np.float32 for v in got.values()) and sum(v.nbytes for v in got.values()) <= 4000
    np.testing.assert_array_equal(got["small"], small.numpy())
    assert got["big"].shape == (500,) and np.isin(got["big"], big.numpy()).all()
    np.testing.assert_array_equal(np.load(tmp_path / "b" / "big.npy"), got["big"])


def test_bench_roofline_traffic_comes_from_the_committed_ncu_extracts():
    """bench.py never types DRAM traffic in: `roofline.traffic` is read from the `metric,unit,value` extracts of `ncu --set full`
    reports committed under profiles/ (tools/ncu_extract.py); a missing capture or a capture of another kernel gives None."""
    import bench
    for csv_name, kernel in (("r02_attn3.ncu.csv", "attn_pnp_kernel"), ("r02_tattn_fused.ncu.csv", "tattn_fused"),
                             ("r02_groupnorm.ncu.csv", "gn_persistent_kernel"), ("r02_gemm_lin960.ncu.csv", "gemm_tcgen05_kernel"),
                             ("r02_gemm_geglu.ncu.csv", "gemm_tcgen05_kernel")):
        got = bench.ncu_traffic((csv_name,), kernel)
        assert got["traffic"] is not None and 1e7 < got["traffic"] < 5e9, (csv_name, got)
        assert csv_name in got["traffic_unit"]
    assert bench.ncu_traffic(("r02_groupnorm.ncu.csv",), "attn_pnp_kernel")["traffic"] is None   # capture of another kernel
    assert bench.ncu_traffic(("no_such_file.csv",), "gemm_tcgen05_kernel")["traffic"] is None


@torch.no_grad()
def test_pipeline_vae_brackets_and_tensor2vid_on_cpu():
    """Host logic of the steps either side of the loops (pipeline_i2vgen_xl.py:79-97, :443-463, :565-592): the pipeline
    delegates to whatever module speaks diffusers' VAE protocol — here the oracle VAE on the CPU — and `tensor2vid`
    reproduces the three output types."""
    import numpy as np
    from anyv2v_b200.pipeline import I2VGenXLPipeline, tensor2vid
    from oracle import vae_ref
    vae = vae_ref.seeded_vae(vae_ref.TINY_VAE_CONFIG, seed=8888)
    pipe = I2VGenXLPipeline(unet=None, vae=vae)
    g = torch.Generator().manual_seed(2)
    lat = torch.randn(1, 4, 2, 4, 6, generator=g)
    video = pipe.decode_latents(lat, decode_chunk_size=1)
    assert video.shape == (1, 3, 2, 8, 12) and video.dtype == torch.float32
    torch.testing.assert_close(video, vae_ref.decode_latents(vae, lat, 1))
    pt = tensor2vid(video, "pt")
    assert pt.shape == (1, 2, 3, 8, 12) and float(pt.min()) >= 0.0 and float(pt.max()) <= 1.0
    arr = tensor2vid(video, "np")
    assert arr.shape == (1, 2, 8, 12, 3) and arr.dtype == np.float32
    np.testing.assert_allclose(arr[0, 1], pt[0, 1].permute(1, 2, 0).numpy(), rtol=0, atol=1e-7)
    pil = tensor2vid(video, "pil")
    assert len(pil) == 1 and len(pil[0]) == 2 and pil[0][0].size == (12, 8)
    with pytest.raises(ValueError, match="does not exist"):
        tensor2vid(video, "mp4")
    frames = torch.randn(2, 3, 8, 8, generator=g).clamp(-1, 1)
    z = pipe.encode_vae_video(frames, generator=torch.Generator().manual_seed(5))
    torch.testing.assert_close(z, vae_ref.encode_vae_video(vae, frames, torch.Generator().manual_seed(5)))
    with pytest.raises(ValueError, match="needs a VAE"):
        I2VGenXLPipeline(unet=None).decode_latents(lat)


def test_attn2q_barrier_protocol_model():
    """tools/protocol_sim.py restates the warp roles of csrc/attention2q_tcgen05.cu (same waits / arrives / commits, same
    parity expressions) and runs them under randomised latencies: no deadlock, no buffer hazard."""
    import random
    from tools import protocol_sim
    rng = random.Random(7)
    for items, n_kv, stages in ((1, 1, 4), (2, 2, 4), (3, 8, 4), (2, 32, 4), (5, 3, 2), (3, 7, 3)):
        for _ in range(6):
            protocol_sim.simulate_attn2q(random.Random(rng.getrandbits(32)), items, n_kv, stages)
    # attn2q_split_kernel: two warps per lane quarter and query tile, row maximum exchanged through double-buffered slots + a named barrier
    for items, n_kv, stages in ((1, 16, 4), (2, 32, 4), (3, 17, 3), (2, 1, 4)):
        for _ in range(4):
            protocol_sim.simulate_attn2q(random.Random(rng.getrandbits(32)), items, n_kv, stages, split=True)
    caught = 0
    for _ in range(10):  # negative control: one exchange buffer instead of two -> a late read sees the partner's NEXT tile
        try:
            protocol_sim.simulate_attn2q(random.Random(rng.getrandbits(32)), 2, 24, 4, split=True, single_xchg_buffer=True)
        except AssertionError:
            caught += 1
    assert caught == 10


def test_fused_temporal_attention_barrier_protocol_model():
    """csrc/attention_tfused_tcgen05.cu: projection ring -> convert -> S -> softmax -> PV with the next item's projection
    issued under the current softmax"""
    import random
    from tools import protocol_sim
    rng = random.Random(5)
    for items, num_kb, stages in ((1, 5, 4), (3, 5, 4), (6, 20, 4), (4, 1, 2), (5, 8, 3)):
        for _ in range(6):
            protocol_sim.simulate_tfused(random.Random(rng.getrandbits(32)), items, num_kb, stages)


def test_two_slot_fused_temporal_attention_barrier_protocol_model():
    """tattn_fused2_kernel: two convert / softmax warpgroups on alternate items, each TMEM slot's accumulator columns re-used in place
    (Q fp16 over Q, S over the K / V accumulators, P over S), MMA order S(i) PV(i-1) QKV(i+1): no deadlock, no aliasing hazard under
    randomised latencies — and the model does catch a wrong order (QKV(i+1) issued before PV(i-1))."""
    import random
    from tools import protocol_sim
    rng = random.Random(11)
    for items, num_kb, stages in ((1, 5, 4), (2, 5, 4), (3, 5, 4), (7, 10, 4), (4, 1, 2), (10, 8, 3)):
        for _ in range(6):
            protocol_sim.simulate_tfused2(random.Random(rng.getrandbits(32)), items, num_kb, stages)
    caught = 0
    for _ in range(10):  # negative control: the projection of item i + 1 issued while PV(i - 1) still owns the slot
        try:
            protocol_sim.simulate_tfused2(random.Random(rng.getrandbits(32)), 6, 5, 4, wrong_order=True)
        except AssertionError:
            caught += 1
    assert caught == 10


def test_lean_gemm_epilogue_bookkeeping_model():
    """tools/epilogue_schedule_model.py restates the counters of the lean GEMM epilogue (division-free tile iterator, chunk ownership of
    the two groups with the alternating odd chunk, residual prefetch cursor, output staging ring + rotating store issuer) and checks
    them against the plain definitions for the tile shapes of the step, ragged N, GEGLU pairs and both staging depths."""
    from tools import epilogue_schedule_model as m
    visits = 0
    for BN, N, geglu in ((160, 960, False), (160, 320, False), (256, 2560, True), (128, 320, False), (64, 200, False), (256, 1280, False),
                         (128, 1280, True), (160, 1000, False)):
        n_tiles = (N + BN - 1) // BN
        for first, stride, m_units in ((0, 148, 1536), (147, 148, 1536), (3, 7, 40), (5, 74, 193), (0, 1, 3)):
            for k_ob in (2, 3):
                visits += m.check(first, stride, m_units, n_tiles, N, BN, geglu, k_ob)
    assert visits > 10000


def test_fma_pipe_exp2_polynomial_emulation():
    """ex2_poly of csrc/ptx.cuh (used by attention2q / attention_v10) emulated in float32 / int32: accuracy far below fp16 resolution, and no
    exponent-field wrap-around for masked keys (-inf) — the clamp must stay at -125 (see the kernel comment)."""
    from tools import exp2_poly_fit
    rel, masked = exp2_poly_fit.check()
    assert rel < 1.0e-4
    assert 0.0 < masked < 6.0e-8  # below the smallest fp16 subnormal: packs to zero
    import re
    src = open(os.path.join(ROOT, "anyv2v_b200", "csrc", "ptx.cuh")).read()
    consts = [float(c) for c in re.findall(r"fmaf\([pf], (?:f, )?([0-9.]+)f", src)] + \
             [float(c) for c in re.findall(r"fmaf\(f, [0-9.]+f, ([0-9.]+)f\)", src)]
    for c in exp2_poly_fit.C:
        assert any(abs(float(c) - k) < 1e-7 for k in consts), f"device constant {float(c)} not found in the kernel source"
    assert "fmaxf(x, -125.0f)" in src


@pytest.mark.parametrize("poly", [0, 1, 2])
def test_attn2q_algorithm_emulation(poly):
    """tools/attn2q_emulation.py: the per-row algorithm of csrc/attention2q_tcgen05.cu (128-key tiles, thresholded running
    max with O / l rescale, fp16 P, FMA-pipe exp2 on 0 / 25 / 50 % of the elements, key-tail masks) against exact softmax
    attention at the tolerance of the GPU parity tests."""
    from tools import attn2q_emulation as em
    for kw in (dict(T=64, L=300), dict(T=128, L=145), dict(T=64, L=512, mag=6.0), dict(T=64, L=640, rising=True)):
        assert em.check(poly=poly, **kw) < 0.5, (poly, kw)

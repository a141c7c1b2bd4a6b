"""GPU tests of non-square frame sizes — I2VGen-XL's native 1280 x 704 (latent 160 x 88) and portrait 704 x 1280: the implicit-GEMM
convolution on block-shaped tiles (edge blocks, residual, row bias, 3-slot injection, stride 2, the Upsample2D phases, CTA pairs)
against fp32 torch, the full-size UNet and the VAE against the oracle, and the two runners end to end."""
import os
from types import SimpleNamespace

import pytest
import torch
import yaml

from parity_utils import assert_fp16_close, err_stats

pytestmark = pytest.mark.gpu
dev = "cuda"


@pytest.fixture(scope="module")
def ops():
    from anyv2v_b200 import ops as o
    return o


def _packed(w):
    return w.permute(0, 2, 3, 1).reshape(w.shape[0], -1).contiguous()


# (NF, H, W, Cin, Cout): widths 160 / 320 / 176 / 352 / 704 / 88 / 20 / 11 / 80 / 40, heights with partial bottom blocks (11, 22, 44),
# Cin >= 128 -> K >= 1152 -> CTA pairs (odd m_tiles included: 11 x 352 is 33 tiles), Cin = 64 -> single CTAs
CONV_GEOS = [(2, 88, 160, 320, 320), (2, 44, 320, 128, 128), (2, 22, 176, 128, 256), (1, 11, 352, 128, 128), (1, 11, 704, 64, 64),
             (3, 160, 88, 320, 320), (3, 11, 20, 640, 640), (4, 20, 11, 320, 320), (2, 44, 80, 640, 640), (2, 22, 40, 1280, 1280),
             (2, 88, 44, 64, 64)]


@pytest.mark.parametrize("geo", CONV_GEOS)
def test_conv3x3_block_tiles(ops, geo):
    NF, H, W, Cin, Cout = geo
    torch.manual_seed(31)
    x = torch.randn(NF, H, W, Cin, device=dev).half()
    w = (torch.randn(Cout, Cin, 3, 3, device=dev) / (9 * Cin) ** 0.5).half()
    bias, temb = torch.randn(Cout, device=dev).half(), torch.randn(NF, Cout, device=dev).half()
    res = torch.randn(NF, H, W, Cout, device=dev).half()
    h = torch.nn.functional.conv2d(x.permute(0, 3, 1, 2).float(), w.float(), bias.float(), padding=1).permute(0, 2, 3, 1)
    out = ops.conv3x3(x, _packed(w), bias=bias, rowbias=temb, rows_per_rowbias=H * W)
    assert_fp16_close(out, h + temb.float()[:, None, None, :], f"conv3x3 block tiles +rowbias {geo}")
    out = ops.conv3x3(x, _packed(w), bias=bias, residual=res)
    assert_fp16_close(out, h + res.float(), f"conv3x3 block tiles +residual {geo}")
    # a tile that ran past the image would write into a neighbouring frame / row: compare the output with the reference to the
    # last element, and check an output buffer with guard rows around it is untouched outside the image
    guard = torch.full((NF * H * W + 256, Cout), 7.0, device=dev, dtype=torch.float16)
    ops.conv3x3(x, _packed(w), bias=bias, out=guard[128:128 + NF * H * W].view(NF, H, W, Cout))
    assert bool((guard[:128] == 7).all()) and bool((guard[128 + NF * H * W:] == 7).all()), f"store outside the image {geo}"


@pytest.mark.parametrize("geo", [(2, 88, 160, 8, 320), (2, 160, 88, 8, 320), (2, 88, 160, 320, 4), (2, 160, 88, 320, 4)])
def test_conv_in_and_conv_out_at_native_resolution(geo):
    """conv_in (8 channels present in a 64-wide K block) and conv_out (4 output channels padded to 8) at latent 160 x 88 / 88 x 160"""
    from anyv2v_b200.unet_i2vgen_xl import Conv3x3
    NF, H, W, Cin, Cout = geo
    torch.manual_seed(32)
    conv = Conv3x3(Cin, Cout).to(device=dev, dtype=torch.float16)
    x = torch.randn(NF, H, W, Cin, device=dev).half()
    got = conv.forward_nhwc(x)
    ref = torch.nn.functional.conv2d(x.float().permute(0, 3, 1, 2), conv.weight.float(), conv.bias.float(), padding=1).permute(0, 2, 3, 1)
    assert got.shape == (NF, H, W, Cout)
    assert_fp16_close(got, ref, f"conv3x3 padded channels {geo}")


@pytest.mark.parametrize("hw", [(22, 40), (40, 22)])
def test_conv3x3_inject_slots_block_tiles(ops, hw):
    """the PnP injection conv (up_blocks[1].resnets[1].conv1 shape: 2560 -> 1280) at the 40 x 22 level: one accumulator tile stored
    to the three branch slots, each with its own residual, through the block map"""
    H, W = hw
    torch.manual_seed(33)
    n, Cin, C = 2, 2560, 1280
    x = torch.randn(n, H, W, Cin, device=dev).half()
    w = (torch.randn(C, Cin, 3, 3, device=dev) / (9 * Cin) ** 0.5).half()
    bias = torch.randn(C, device=dev).half()
    short = torch.randn(3, n, H, W, C, device=dev).half()
    out = torch.empty_like(short)
    ops.conv3x3(x, _packed(w), bias=bias, residual=short, out=out, n_slots=3, slot_stride=n * H * W * C)
    h = torch.nn.functional.conv2d(x.permute(0, 3, 1, 2).float(), w.float(), bias.float(), padding=1).permute(0, 2, 3, 1)
    assert_fp16_close(out, h[None] + short.float(), f"conv3x3 3-slot {hw}")


@pytest.mark.parametrize("geo", [(2, 88, 160, 320, 320), (2, 160, 88, 320, 320), (1, 176, 320, 128, 128), (1, 22, 40, 640, 640)])
def test_conv3x3_stride2_block_tiles(ops, geo):
    """Downsample2D from 160 x 88 / 88 x 160 (outputs 80 x 44 / 44 x 80 on 16 x 8 blocks) and wider / ragged inputs"""
    NF, H, W, Cin, Cout = geo
    torch.manual_seed(34)
    x = torch.randn(NF, H, W, Cin, device=dev).half()
    w = (torch.randn(Cout, Cin, 3, 3, device=dev) / (9 * Cin) ** 0.5).half()
    b = (0.1 * torch.randn(Cout, device=dev)).half()
    got = ops.conv3x3(x, _packed(w), bias=b, stride=2)
    ref = torch.nn.functional.conv2d(x.float().permute(0, 3, 1, 2), w.float(), b.float(), stride=2, padding=1).permute(0, 2, 3, 1)
    assert got.shape == (NF, H // 2, W // 2, Cout)
    assert_fp16_close(got, ref, f"conv3x3 stride 2 {geo}")


@pytest.mark.parametrize("geo", [(2, 11, 20, 1280), (2, 22, 40, 1280), (2, 44, 80, 640), (2, 20, 11, 1280), (2, 40, 22, 1280),
                                 (2, 80, 44, 640)])
def test_upsample2x_conv3x3_block_tiles(ops, geo):
    """the four Upsample2D phases on block tiles whose last block ends inside a frame (20 x 6 blocks at 20 x 11, ...): the 5-D store
    map clips the block at the frame's last row instead of writing into the next frame"""
    NF, H, W, C = geo
    torch.manual_seed(35)
    x = torch.randn(NF, H, W, C, device=dev).half()
    w = (torch.randn(C, C, 3, 3, device=dev) / (9 * C) ** 0.5).half()
    b = (0.1 * torch.randn(C, device=dev)).half()
    got = ops.upsample2x_conv3x3(x, ops.pack_upsample_weights(w), bias=b)
    up = torch.nn.functional.interpolate(x.float().permute(0, 3, 1, 2), scale_factor=2.0, mode="nearest")
    ref = torch.nn.functional.conv2d(up, w.float(), b.float(), padding=1).permute(0, 2, 3, 1)
    assert got.shape == (NF, 2 * H, 2 * W, C)
    assert_fp16_close(got, ref, f"fused upsample conv {geo}", atol_frac=2e-3)


# ------------------------------------------------------------------------------------------------ full-size UNet vs the oracle
SIZES = [(88, 160), (160, 88)]  # latent (h, w): 1280 x 704 and 704 x 1280 frames
F2 = 2


@pytest.fixture(scope="module")
def full():
    import test_gpu_fullwidth as fw
    return fw.build_models(dev)


@torch.no_grad()
@pytest.mark.parametrize("hw", SIZES)
def test_fullsize_unet_hooked_step_native_resolution(full, hw):
    """one hooked step (conv + spatial + temporal injection fire at t = 901), B = 3 branches, F = 2 frames"""
    import test_gpu_fullwidth as fw
    from anyv2v_b200 import ops
    H, W = hw
    _, schedule = fw._schedule()
    fw._register(full, schedule, 901)
    outs = {}
    c0 = ops.launch_count()
    for name, net, dt in (("ours", full.ours, torch.float16), ("ref32", full.ref32, torch.float32), ("ref16", full.ref16, torch.float16)):
        _, x3, prompts, img_lat, img_emb, fps = fw._inputs(dt, F=F2, H=H, W=W)
        outs[name] = net(x3, torch.tensor([901], device=dev), fps, img_lat, img_emb, prompts)[0]
    assert ops.launch_count() - c0 > 500
    assert outs["ours"].shape == (3, 4, F2, H, W)
    fw._check(outs["ours"], outs["ref32"], outs["ref16"], f"full-size hooked UNet step at latent {W}x{H}")
    fw._register(full, [], -1)


@torch.no_grad()
@pytest.mark.parametrize("hw", SIZES)
def test_fullsize_unet_forward_b1_native_resolution(full, hw):
    import test_gpu_fullwidth as fw
    H, W = hw
    fw._register(full, [], -1)
    outs = {}
    for name, net, dt in (("ours", full.ours, torch.float16), ("ref32", full.ref32, torch.float32), ("ref16", full.ref16, torch.float16)):
        ns, _, _, _, _, _ = fw._inputs(dt, F=F2, H=H, W=W)
        outs[name] = net(ns.video_latents, torch.tensor([21], device=dev), ns.fps, ns.src_image_latents, ns.src_image_emb, ns.inv_prompt)[0]
    fw._check(outs["ours"], outs["ref32"], outs["ref16"], f"full-size B=1 forward at latent {W}x{H}")


@torch.no_grad()
@pytest.mark.parametrize("hw", SIZES)
def test_fullsize_pipeline_steps_native_resolution(full, hw):
    """one teacher-forced inversion iteration and one edit iteration (all three injections fire) through the product pipeline
    against the oracle; then the same iterations replayed from captured CUDA graphs are bit-identical to the eager launches"""
    import test_gpu_fullwidth as fw
    from anyv2v_b200.latent_store import LatentStore
    from anyv2v_b200.pipeline import I2VGenXLPipeline
    from anyv2v_b200.run_group_pnp_edit import init_pnp
    from anyv2v_b200.schedulers import DDIMInverseScheduler, DDIMScheduler
    from oracle import loops_ref, pnp_hooks_ref, schedulers_ref
    H, W = hw
    n_steps = 50
    ns32, _, _, _, _, _ = fw._inputs(torch.float32, F=F2, H=H, W=W)
    ns16, _, _, _, _, _ = fw._inputs(torch.float16, F=F2, H=H, W=W)
    fw._register(full, [], -1)
    # ---- inversion, first iteration
    inv_ref = schedulers_ref.DDIMInverseScheduler()
    inv_ref.set_timesteps(n_steps)
    t = int(inv_ref.timesteps[0])
    x32 = ns32.video_latents
    v = full.ref32(x32, torch.tensor([t], device=dev), ns32.fps, ns32.src_image_latents, ns32.src_image_emb, ns32.inv_prompt)[0]
    want, _ = inv_ref.step(v, t, x32)
    v16 = full.ref16(x32.half(), torch.tensor([t], device=dev), ns16.fps, ns16.src_image_latents, ns16.src_image_emb, ns16.inv_prompt)[0]
    want16, _ = inv_ref.step(v16, t, x32.half())
    pipe = I2VGenXLPipeline(full.ours, DDIMInverseScheduler())
    runs = []
    for graphs in (False, True, True, True):  # eager, then first use / capture / replay of the graphed iteration
        pipe.use_cuda_graphs = graphs
        if not runs or len(runs) == 1:
            st = pipe.prepare_invert(ns16.video_latents, ns16.inv_prompt, ns16.src_image_latents, ns16.src_image_emb, 8, n_steps,
                                     1.0, None, False, False)
        st.latents.copy_(x32.half())
        runs.append(pipe.invert_step(st, 0).clone())
    fw._check(runs[0], want, want16, f"teacher-forced inversion step t={t} at latent {W}x{H}")
    assert torch.equal(runs[0], runs[-1]) and torch.equal(runs[0], runs[-2]), "inversion: graph replay differs from eager"
    # ---- edit, first iteration (conv + spatial + temporal injection)
    sref = schedulers_ref.DDIMScheduler()
    sref.set_timesteps(n_steps)
    for net in (full.ref32, full.ref16):
        pnp_hooks_ref.init_pnp(SimpleNamespace(unet=net), sref, n_steps, 0.8, 0.5, 0.5)
    sch = DDIMScheduler()
    sch.set_timesteps(n_steps)
    pipe.register_modules(scheduler=sch)
    init_pnp(pipe, sch, SimpleNamespace(n_steps=n_steps, pnp_f_t=0.8, pnp_spatial_attn_t=0.5, pnp_temp_attn_t=0.5))
    prompts, img_lat, img_emb, fps = loops_ref.edit_conditioning(ns32)
    prompts16, img_lat16, img_emb16, fps16 = loops_ref.edit_conditioning(ns16)
    g = torch.Generator().manual_seed(78)
    t = int(sref.timesteps[0])
    src = torch.randn(1, 4, F2, H, W, generator=g).to(dev)
    x = torch.randn(1, 4, F2, H, W, generator=g).to(dev)
    pnp_hooks_ref.register_time(SimpleNamespace(unet=full.ref32), t)
    v = full.ref32(torch.cat([src, x, x]), torch.tensor([t], device=dev), fps, img_lat, img_emb, prompts)[0]
    want, _ = sref.step(schedulers_ref.cfg_combine(v[1:2], v[2:3], 9.0), t, x)
    pnp_hooks_ref.register_time(SimpleNamespace(unet=full.ref16), t)
    v16 = full.ref16(torch.cat([src, x, x]).half(), torch.tensor([t], device=dev), fps16, img_lat16, img_emb16, prompts16)[0]
    want16, _ = sref.step(schedulers_ref.cfg_combine(v16[1:2], v16[2:3], 9.0), t, x.half())
    store = LatentStore(None, write_files=False)
    store.put(t, src.half())
    runs = []
    for graphs in (False, True, True, True):
        pipe.use_cuda_graphs = graphs
        if len(runs) <= 1:
            st_e = pipe.prepare_edit(x.half(), ns16.edit_prompt, ns16.neg_prompt, ns16.inv_prompt, ns16.edit_image_emb,
                                     ns16.edit_image_latents, ns16.src_image_emb, ns16.src_image_latents, 8, n_steps, 9.0, 0, None,
                                     store, True)
        st_e.latents.copy_(x.half())
        runs.append(pipe.edit_step(st_e, 0).clone())
    assert pipe._hook_flags(t) == (True, True, True)
    fw._check(runs[0], want, want16, f"teacher-forced PnP edit step t={t} at latent {W}x{H}")
    assert torch.equal(runs[0], runs[-1]) and torch.equal(runs[0], runs[-2]), "edit: graph replay differs from eager"
    fw._register(full, [], -1)


# ------------------------------------------------------------------------------------------------ VAE (SD KL-f8 config) vs the oracle
@pytest.fixture(scope="module")
def sd_vaes():
    from anyv2v_b200 import vae as product
    from oracle import vae_ref
    ref32 = vae_ref.seeded_vae(vae_ref.SD_VAE_CONFIG, seed=8888, dtype=torch.float32).to(dev)
    ref16 = vae_ref.seeded_vae(vae_ref.SD_VAE_CONFIG, seed=8888, dtype=torch.float16).to(dev)
    ours = product.AutoencoderKL(**vae_ref.SD_VAE_CONFIG)
    ours.load_state_dict(ref32.state_dict())
    ours = ours.to(device=dev, dtype=torch.float16).eval()
    return SimpleNamespace(ref32=ref32, ref16=ref16, ours=ours)


def _close_as_fp16_torch(got, ref32, ref16, what, slack=3.0):
    assert torch.isfinite(got).all(), what
    e_ours, e_ref = err_stats(got, ref32), err_stats(ref16, ref32)
    print(f"{what}: ours-vs-fp32 {e_ours}  |  torch-fp16-vs-fp32 {e_ref}")
    assert e_ours["rms_rel"] <= max(slack * e_ref["rms_rel"], 2e-3), (what, e_ours, e_ref)


@torch.no_grad()
@pytest.mark.parametrize("size", [(1280, 704), (704, 1280)])
def test_vae_native_resolution_matches_oracle(sd_vaes, size):
    from anyv2v_b200 import vae as product
    from oracle import vae_ref
    Wp, Hp = size
    g = torch.Generator().manual_seed(13)
    frames = torch.randn(1, 3, Hp, Wp, generator=g).clamp(-1, 1).to(dev)
    d32 = sd_vaes.ref32.encode(frames.float()).latent_dist
    d16 = sd_vaes.ref16.encode(frames.half()).latent_dist
    dours = sd_vaes.ours.encode(frames.half()).latent_dist
    assert dours.mean.shape == (1, 4, Hp // 8, Wp // 8)
    _close_as_fp16_torch(dours.mean, d32.mean, d16.mean, f"vae posterior mean {Wp}x{Hp}")
    lat = torch.randn(1, 4, 2, Hp // 8, Wp // 8, generator=g).to(dev)
    ref32 = vae_ref.decode_latents(sd_vaes.ref32, lat.float(), 1)
    ref16 = vae_ref.decode_latents(sd_vaes.ref16, lat.half(), 1)
    got = product.decode_latents(sd_vaes.ours, lat.half(), None)
    assert got.shape == ref32.shape == (1, 3, 2, Hp, Wp)
    _close_as_fp16_torch(got, ref32, ref16, f"vae decode {Wp}x{Hp}")


# ------------------------------------------------------------------------------------------------ runners at image_size [1280, 704]
def test_group_runners_at_1280x704(tmp_path):
    """run_group_ddim_inversion -> run_group_pnp_edit on real png frames with `image_size: [1280, 704]` (the reference template's
    native size), tiny UNet / VAE / CLIP towers: latents [.., 88, 160] on disk, 1280 x 704 png / gif out"""
    import test_gpu_runners as gr
    from anyv2v_b200 import run_group_ddim_inversion as inv, run_group_pnp_edit as edit
    from anyv2v_b200.config import OmegaConf
    from oracle.unet_ref import TINY_CONFIG
    from PIL import Image
    torch.set_grad_enabled(False)
    device = torch.device("cuda", 0)
    data = str(tmp_path)
    edited = gr.write_demo_clip(data, n=2, size=(1280, 704))
    size = [1280, 704]
    inv_t = dict(gr.INV_TEMPLATE, data_dir=data, device=str(device), synthetic=False, image_size=size, n_frames=2)
    inv_t["inverse_config"] = dict(inv_t["inverse_config"], n_steps=2, prompt="a man", negative_prompt="blurry")
    inv_t["recon_config"] = dict(inv_t["recon_config"], enable_recon=False)
    (tmp_path / "inv.yaml").write_text(yaml.safe_dump(inv_t))
    (tmp_path / "edit.yaml").write_text(yaml.safe_dump(dict(gr.EDIT_TEMPLATE, data_dir=data, device=str(device), synthetic=False,
                                                            image_size=size, n_frames=2, n_steps=2)))
    entries = [{"active": True, "video_name": "clipA", "edited_first_frame_path": edited, "editing_prompt": "a robot",
                "edited_video_name": "robot", "ddim_init_latents_t_idx": 0, "pnp_f_t": 1.0, "pnp_spatial_attn_t": 1.0, "pnp_temp_attn_t": 1.0}]
    kw = dict(vae_config=gr.TINY_VAE)
    out = inv.main(OmegaConf.load(str(tmp_path / "inv.yaml")), entries, device, unet_config=TINY_CONFIG, pipeline_kwargs=kw)
    assert len(out) == 1 and out[0].shape == (2, 4, 2, 88, 160) and torch.isfinite(out[0]).all()
    lat_dir = os.path.join(data, "inversions", "i2vgen-xl", "clipA", "ddim_latents")
    files = sorted(os.listdir(lat_dir))
    assert len(files) == 2 and torch.load(os.path.join(lat_dir, files[0]), map_location="cpu").shape == (1, 4, 2, 88, 160)
    res = edit.main(OmegaConf.load(str(tmp_path / "edit.yaml")), entries, device, unet_config=TINY_CONFIG, pipeline_kwargs=kw)
    assert len(res) == 1 and res[0].shape == (1, 4, 2, 88, 160) and torch.isfinite(res[0]).all()
    od = os.path.join(data, "Results", "Prompt-Based-Editing", "i2vgen-xl", "clipA", "robot",
                      "ddim_init_latents_t_idx_0_nsteps_2_cfg_9.0_pnpf1.0_pnps1.0_pnpt1.0")
    names = set(os.listdir(od))
    assert {"video.gif", "edited_latents.pt", "video_00000.png", "video_00001.png"} <= names, names
    assert Image.open(os.path.join(od, "video_00001.png")).size == (1280, 704)

"""Shape census of one UNet step WITHOUT a GPU: the full-size I2VGen-XL UNet is built on the meta device, anyv2v_b200.ops is
replaced by shape-only stubs, and every kernel call of an inversion step (B = 1) and a PnP edit step (B = 3, conv + spatial
injection) at 16 frames x 64 x 64 latents is recorded.  For every GEMM the tile plan of csrc/gemm_tcgen05.cu's cost model is
re-derived (same formula) and the wave quantisation on 148 SMs is reported:

    python tools/shape_census.py            # table: calls, FLOPs, tiles, waves, efficiency, share of the step's GEMM FLOPs
"""
from __future__ import annotations

import math
import os
import sys
from collections import OrderedDict
from types import SimpleNamespace

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
SMS = 148


def plan(M, N, K, mode, geglu, m_tiles):
    """tile-N choice of av2v_gemm_f16 (gemm_tcgen05.cu) and the pair-mode rule"""
    best, bn = None, 0
    for c in (256, 160, 128, 64):
        if N % c:
            continue
        if geglu and (c // 32) % 2:
            continue
        tiles = m_tiles * (N // c)
        waves = -(-tiles // SMS)
        l2 = (128 + c) * 4 // 5
        cost = waves * (max(c, l2) + 32)
        if best is None or cost < best:
            best, bn = cost, c
    if bn == 0:
        bn = 128 if N > 256 else 64
    n_tiles = -(-N // bn)
    num_kb = {"linear": -(-K // 64), "conv3x3": K // 64, "tconv3": K // 64}[mode]
    pair = num_kb >= 10 and m_tiles >= 2 and N % bn == 0
    if pair:
        units, slots = -(-m_tiles // 2) * n_tiles, SMS // 2
    else:
        units, slots = m_tiles * n_tiles, SMS
    waves = units / slots
    eff = waves / math.ceil(waves)
    return bn, pair, units, waves, eff


def census(batch, inject):
    from anyv2v_b200 import ops, pnp_utils
    from anyv2v_b200.unet_i2vgen_xl import I2VGEN_XL_CONFIG, I2VGenXLUNet
    calls = []
    empty = lambda shape, like: torch.empty(shape, dtype=torch.float16, device=like.device)

    def linear(a, w, bias=None, residual=None, out=None, rowbias=None, rows_per_rowbias=0, geglu=False):
        M, K = a.shape
        N = w.shape[0]
        calls.append(("linear" + ("+geglu" if geglu else "") + ("+res" if residual is not None else ""), "linear", M, N, K, (M + 127) // 128, geglu))
        return out if out is not None else empty((M, N // 2 if geglu else N), a)

    def conv3x3(x, w, bias=None, rowbias=None, rows_per_rowbias=0, residual=None, out=None, n_slots=1, slot_stride=0):
        NF, H, W, Cin = x.shape
        Cout = w.shape[0]
        M = NF * H * W
        hw = H * W
        m_tiles = NF * (-(-H // max(1, min(H, 128 // W)))) if hw >= 128 else -(-NF // (128 // hw))
        calls.append(("conv3x3" + ("+res" if residual is not None else "") + (f"+slots{n_slots}" if n_slots > 1 else ""), "conv3x3", M, Cout, 9 * Cin, m_tiles, False))
        return out if out is not None else empty((NF, H, W, Cout), x)

    def tconv3(x, w, F, HW, bias=None, residual=None, out=None):
        B, R, Cin = x.shape
        Cout = w.shape[0]
        calls.append(("tconv3" + ("+res" if residual is not None else ""), "tconv3", B * R, Cout, 3 * Cin, B * (-(-R // 128)), False))
        return out if out is not None else empty((B, R, Cout), x)

    def groupnorm(x, g, b, groups, eps, silu, out=None):
        calls.append(("groupnorm" + ("+silu" if silu else ""), "gn", x.shape[0], x.shape[1], x.shape[2], 0, False))
        return torch.empty_like(x)

    def layernorm(x, g, b, eps=1e-5, out=None):
        calls.append(("layernorm", "ln", x.numel() // x.shape[-1], x.shape[-1], 0, 0, False))
        return torch.empty_like(x)

    def attention(q, k, v, heads, seq, batch, out, scale=0.125, n_v=1, v_branch_stride=0, o_branch_stride=0, frames_mode=False,
                  HW=0, seq_kv=0, kv_batch_div=0):
        calls.append((f"attention {'frames' if frames_mode else 'rows'} nv={n_v}", "attn", batch, seq, seq_kv or seq, heads, False))
        return out

    saved = {n: getattr(ops, n) for n in ("linear", "conv3x3", "tconv3", "groupnorm", "layernorm", "attention")}
    for n, f in dict(linear=linear, conv3x3=conv3x3, tconv3=tconv3, groupnorm=groupnorm, layernorm=layernorm, attention=attention).items():
        setattr(ops, n, f)
    try:
        with torch.device("meta"):
            net = I2VGenXLUNet(**I2VGEN_XL_CONFIG).half()
        F_, H_, W_ = 16, 64, 64
        m = lambda *s: torch.empty(*s, dtype=torch.float16, device="meta")
        pipe = SimpleNamespace(unet=net)
        if inject:
            pnp_utils.register_conv_injection(pipe, [981])
            pnp_utils.register_spatial_attention_pnp(pipe, [981])
            pnp_utils.register_temp_attention_pnp(pipe, [])
            pnp_utils.register_time(pipe, 981)
        cond = dict(fps_emb=m(batch, 1280), ctx=m(batch, 145, 1024), image_latents_nhwc=m(batch * F_, H_, W_, 4))
        with torch.no_grad():
            net(m(batch, 4, F_, H_, W_), torch.empty(1, dtype=torch.int64, device="meta"), cond=cond)
    finally:
        for n, f in saved.items():
            setattr(ops, n, f)
    return calls


def _conv_stubs(convs):
    """shape-only stand-ins for every anyv2v_b200.ops entry the UNet / VAE forward passes call; the 3x3 convolutions (plain,
    strided and the four phases of the fused Upsample2D) are recorded as av2v_gemm_args field dicts"""
    empty = lambda shape, like: torch.empty(shape, dtype=torch.float16, device=like.device)

    def linear(a, w, bias=None, residual=None, out=None, rowbias=None, rows_per_rowbias=0, geglu=False, a2=None):
        return out if out is not None else empty((a.shape[0], w.shape[0] // 2 if geglu else w.shape[0]), a)

    def conv3x3(x, w, bias=None, rowbias=None, rows_per_rowbias=0, residual=None, out=None, n_slots=1, slot_stride=0, stride=1):
        NF, H, W, C = x.shape
        Cout, Cin = w.shape[0], w.shape[1] // 9
        convs.append(dict(NF=NF, H=H, W=W, Cin=Cin, N=Cout, K=9 * Cin, M=NF * (H // stride) * (W // stride), stride=stride,
                          a_channels=C if C != Cin else 0, ldo=Cout, n_slots=n_slots, residual=residual is not None,
                          rowbias=rowbias is not None, up2_phase=0))
        return out if out is not None else empty((NF, H // stride, W // stride, Cout), x)

    def upsample2x_conv3x3(x, w_phases, bias=None, out=None):
        NF, H, W, Cin = x.shape
        Cout = w_phases.shape[1]
        for ph in range(4):
            convs.append(dict(NF=NF, H=H, W=W, Cin=Cin, N=Cout, K=4 * Cin, M=NF * H * W, stride=1, a_channels=0, ldo=Cout, n_slots=1,
                              residual=False, rowbias=False, up2_phase=ph + 1))
        return out if out is not None else empty((NF, 2 * H, 2 * W, Cout), x)

    def tconv3(x, w, F, HW, bias=None, residual=None, out=None):
        return out if out is not None else empty((x.shape[0], x.shape[1], w.shape[0]), x)

    def groupnorm(x, g, b, groups, eps, silu, out=None, x2=None):
        return empty(x.shape[:-1] + (x.shape[-1] + (x2.shape[-1] if x2 is not None else 0),), x)

    def layernorm(x, g, b, eps=1e-5, out=None):
        return torch.empty_like(x)

    def attention(q, k, v, heads, seq, batch, out, **kw):
        return out

    def temporal_attention_fused(x, wqkv, heads, F, HW, clips, out, **kw):
        return out

    return dict(linear=linear, conv3x3=conv3x3, upsample2x_conv3x3=upsample2x_conv3x3, tconv3=tconv3, groupnorm=groupnorm,
                layernorm=layernorm, attention=attention, temporal_attention_fused=temporal_attention_fused)


def _with_stubs(convs, fn):
    from anyv2v_b200 import ops
    stubs = _conv_stubs(convs)
    saved = {n: getattr(ops, n) for n in stubs}
    for n, f in stubs.items():
        setattr(ops, n, f)
    try:
        with torch.no_grad():
            fn()
    finally:
        for n, f in saved.items():
            setattr(ops, n, f)
    return convs


def unet_conv_census(batch, inject, frames, height, width):
    """every 3x3 convolution of one full-size UNet forward at latent height x width: an inversion step (batch 1) or a PnP edit
    step (batch 3, conv + spatial injection firing)"""
    from anyv2v_b200 import pnp_utils
    from anyv2v_b200.unet_i2vgen_xl import I2VGEN_XL_CONFIG, I2VGenXLUNet

    def run():
        with torch.device("meta"):
            net = I2VGenXLUNet(**I2VGEN_XL_CONFIG).half()
        m = lambda *s: torch.empty(*s, dtype=torch.float16, device="meta")
        if inject:
            pipe = SimpleNamespace(unet=net)
            pnp_utils.register_conv_injection(pipe, [981])
            pnp_utils.register_spatial_attention_pnp(pipe, [981])
            pnp_utils.register_temp_attention_pnp(pipe, [981])
            pnp_utils.register_time(pipe, 981)
        cond = dict(fps_emb=m(batch, 1280), ctx=m(batch, 145, 1024), image_latents_nhwc=m(batch * frames, height, width, 4))
        net(m(batch, 4, frames, height, width), torch.empty(1, dtype=torch.int64, device="meta"), cond=cond)
    return _with_stubs([], run)


def vae_conv_census(frames, height, width):
    """every 3x3 convolution the VAE runs on the tensor cores for an encode of `frames` height x width frames and the decode
    of their latents"""
    from anyv2v_b200.vae import SD_VAE_CONFIG, AutoencoderKL

    def run():
        with torch.device("meta"):
            vae = AutoencoderKL(**SD_VAE_CONFIG).half()
        vae.encode(torch.empty(frames, 3, height, width, dtype=torch.float16, device="meta"))
        vae.decode(torch.empty(frames, 4, height // 8, width // 8, dtype=torch.float16, device="meta"))
    return _with_stubs([], run)


def report(title, calls):
    gemms = OrderedDict()
    for name, mode, M, N, K, m_tiles, geglu in calls:
        if mode in ("linear", "conv3x3", "tconv3"):
            key = (name, mode, M, N, K, m_tiles, geglu)
            gemms[key] = gemms.get(key, 0) + 1
    total = sum(2.0 * k[2] * k[3] * k[4] * n for k, n in gemms.items())
    print(f"== {title}: {sum(gemms.values())} GEMM launches, {total / 1e12:.2f} TFLOP executed; {len(calls)} kernel calls in all")
    print(f"{'op':22s} {'M':>7s} {'N':>6s} {'K':>6s} calls  GFLOP  share   BN pair  units  waves   eff   lost")
    lost_total = 0.0
    rows = []
    for (name, mode, M, N, K, m_tiles, geglu), n in gemms.items():
        fl = 2.0 * M * N * K * n
        bn, pair, units, waves, eff = plan(M, N, K, mode, geglu, m_tiles)
        lost = fl / total * (1 - eff)
        lost_total += lost
        rows.append((fl, f"{name:22s} {M:7d} {N:6d} {K:6d} {n:5d} {fl / 1e9:6.0f} {fl / total * 100:5.1f}% {bn:4d} {'yes' if pair else ' no'} {units:6d} {waves:6.2f} {eff * 100:5.1f}% {lost * 100:5.2f}%"))
    for _, line in sorted(rows, reverse=True)[:28]:
        print(line)
    print(f"FLOP-weighted wave-quantisation loss over all GEMMs of the step: {lost_total * 100:.1f} %")


if __name__ == "__main__":
    report("inversion step (B = 1)", census(1, False))
    report("PnP edit step (B = 3, conv + spatial injection)", census(3, True))

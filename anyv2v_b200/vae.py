"""AutoencoderKL (the KL-f8 VAE of `ali-vilab/i2vgen-xl`) on the hand-written sm_100a kernels — SURVEY §8f row 4: the
steps either side of the sampling loops, `encode_vae_video` (i2vgen-xl/pipelines/pipeline_i2vgen_xl.py:565-592) and
`decode_latents` (:443-463).

Module / parameter names are diffusers' (`encoder.down_blocks.0.resnets.0.norm1.weight`, `decoder.mid_block.attentions.0.to_q…`,
`quant_conv`, `post_quant_conv`), so a real `diffusion_pytorch_model` state_dict loads unchanged.  Activations are
channels-last fp16 end to end; every 3x3 convolution with Cin % 64 == 0 (all but `conv_in`), every GroupNorm(+SiLU),
the 1x1 shortcuts and the attention projections run on `anyv2v_b200.ops` (tcgen05 implicit GEMM, fused bias/residual
epilogue; a conv tile is a block of up to 128 pixels of one frame — 128-pixel row segments at widths that are multiples of
128, 64 x 2 blocks at width 320, 32 x 4 at 160 — so any frame whose sides are multiples of 64 px runs).  Left on library calls for now
(`next_rows`): `conv_in` (3 -> 128), the convolutions that end in 3 / 8 / 4 channels, the stride-2 down-sampling
convolutions, and the single-head 512-wide mid-block attention core (head_dim 512 is outside the d = 64 kernel).
There is no CPU path.

Unlike the reference, which encodes and decodes one frame per VAE call (`decode_chunk_size=1`, one `vae.encode` per
frame), all frames go through in one batch — the per-frame results are identical (every op is per-sample).
"""
from __future__ import annotations

from types import SimpleNamespace
from typing import Sequence

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import next_rows as nr
from . import ops
from .unet_i2vgen_xl import Conv3x3, GroupNorm, Linear, to_nchw_view, to_nhwc

SD_VAE_CONFIG = dict(in_channels=3, out_channels=3, latent_channels=4, block_out_channels=(128, 256, 512, 512),
                     layers_per_block=2, norm_num_groups=32, scaling_factor=0.18215)


class LibConv2d(nn.Conv2d):
    """The VAE's stem / head convolutions (3 -> 128, 128 -> 3 / 8, 4 -> 512 channels) stay on cuDNN: they run once per clip,
    outside the denoising loops, and their channel counts (3) are below the 16-byte granularity of the TMA taps."""

    def forward_nhwc(self, x):
        return nr.conv2d_nhwc(x, self.weight, self.bias, stride=self.stride[0], padding=self.padding[0])

    def forward(self, x):
        return to_nchw_view(self.forward_nhwc(to_nhwc(x)))


class VaeResnetBlock2D(nn.Module):
    """GN -> SiLU -> conv1 -> GN -> SiLU -> conv2 (+ shortcut in the epilogue); no time embedding."""

    def __init__(self, in_channels, out_channels, groups=32, eps=1e-6):
        super().__init__()
        self.in_channels, self.out_channels = in_channels, out_channels
        self.norm1 = GroupNorm(groups, in_channels, eps=eps)
        self.conv1 = Conv3x3(in_channels, out_channels)
        self.norm2 = GroupNorm(groups, out_channels, eps=eps)
        self.conv2 = Conv3x3(out_channels, out_channels)
        self.conv_shortcut = nn.Conv2d(in_channels, out_channels, 1) if in_channels != out_channels else None

    def forward_nhwc(self, x):
        n, h, w, cin = x.shape
        short = x
        if self.conv_shortcut is not None:
            short = ops.linear(x.view(-1, cin), self.conv_shortcut.weight.view(self.out_channels, cin),
                               bias=self.conv_shortcut.bias).view(n, h, w, self.out_channels)
        y = self.norm1.forward_rows(x.view(n, h * w, cin), silu=True).view(n, h, w, cin)
        y = self.conv1.forward_nhwc(y)
        y = self.norm2.forward_rows(y.view(n, h * w, -1), silu=True).view(n, h, w, -1)
        return self.conv2.forward_nhwc(y, residual=short)


class VaeAttention(nn.Module):
    """GroupNorm -> fused q,k,v projection -> one 512-wide head -> out projection with the residual in its epilogue."""

    def __init__(self, channels, groups=32, eps=1e-6):
        super().__init__()
        self.group_norm = GroupNorm(groups, channels, eps=eps)
        self.to_q = Linear(channels, channels)
        self.to_k = Linear(channels, channels)
        self.to_v = Linear(channels, channels)
        self.to_out = nn.ModuleList([Linear(channels, channels), nn.Dropout(0.0)])
        self.heads = 1

    def forward_nhwc(self, x):
        n, h, w, c = x.shape
        rows = x.view(n, h * w, c)
        y = self.group_norm.forward_rows(rows, silu=False)
        wqkv = torch.cat([self.to_q.weight, self.to_k.weight, self.to_v.weight], dim=0)
        bqkv = torch.cat([self.to_q.bias, self.to_k.bias, self.to_v.bias], dim=0)
        qkv = ops.linear(y.view(-1, c), wqkv, bias=bqkv).view(n, h * w, 3 * c)
        o = nr.cross_attention(qkv[..., :c], qkv[..., c:2 * c], qkv[..., 2 * c:], heads=1)  # library SDPA, head_dim = C
        o = ops.linear(o.reshape(-1, c), self.to_out[0].weight, bias=self.to_out[0].bias, residual=rows.reshape(-1, c))
        return o.view(n, h, w, c)


class _Down(nn.Module):
    def __init__(self, channels):
        super().__init__()
        self.conv = nn.Conv2d(channels, channels, 3, stride=2, padding=0)

    def forward_nhwc(self, x):  # diffusers Downsample2D(padding=0): zero pad right / bottom, then stride 2
        return nr.conv2d_nhwc(F.pad(x, (0, 0, 0, 1, 0, 1)), self.conv.weight, self.conv.bias, stride=2, padding=0)


class _Up(nn.Module):
    def __init__(self, channels):
        super().__init__()
        self.conv = Conv3x3(channels, channels)

    def forward_nhwc(self, x):
        return self.conv.forward_nhwc(nr.nearest_up2_nhwc(x))


class DownEncoderBlock2D(nn.Module):
    def __init__(self, cin, cout, layers, groups, add_downsample):
        super().__init__()
        self.resnets = nn.ModuleList([VaeResnetBlock2D(cin if i == 0 else cout, cout, groups) for i in range(layers)])
        self.downsamplers = nn.ModuleList([_Down(cout)]) if add_downsample else None

    def forward_nhwc(self, x):
        for r in self.resnets:
            x = r.forward_nhwc(x)
        if self.downsamplers is not None:
            x = self.downsamplers[0].forward_nhwc(x)
        return x


class UpDecoderBlock2D(nn.Module):
    def __init__(self, cin, cout, layers, groups, add_upsample):
        super().__init__()
        self.resnets = nn.ModuleList([VaeResnetBlock2D(cin if i == 0 else cout, cout, groups) for i in range(layers)])
        self.upsamplers = nn.ModuleList([_Up(cout)]) if add_upsample else None

    def forward_nhwc(self, x):
        for r in self.resnets:
            x = r.forward_nhwc(x)
        if self.upsamplers is not None:
            x = self.upsamplers[0].forward_nhwc(x)
        return x


class UNetMidBlock2D(nn.Module):
    def __init__(self, channels, groups):
        super().__init__()
        self.resnets = nn.ModuleList([VaeResnetBlock2D(channels, channels, groups), VaeResnetBlock2D(channels, channels, groups)])
        self.attentions = nn.ModuleList([VaeAttention(channels, groups)])

    def forward_nhwc(self, x):
        return self.resnets[1].forward_nhwc(self.attentions[0].forward_nhwc(self.resnets[0].forward_nhwc(x)))


class Encoder(nn.Module):
    def __init__(self, in_channels, latent_channels, chans: Sequence[int], layers, groups):
        super().__init__()
        self.conv_in = LibConv2d(in_channels, chans[0], 3, padding=1)
        self.down_blocks = nn.ModuleList()
        c = chans[0]
        for i, co in enumerate(chans):
            self.down_blocks.append(DownEncoderBlock2D(c, co, layers, groups, add_downsample=i < len(chans) - 1))
            c = co
        self.mid_block = UNetMidBlock2D(c, groups)
        self.conv_norm_out = GroupNorm(groups, c, eps=1e-6)
        self.conv_act = nn.SiLU()
        self.conv_out = LibConv2d(c, 2 * latent_channels, 3, padding=1)

    def forward_nhwc(self, x):
        x = self.conv_in.forward_nhwc(x)
        for blk in self.down_blocks:
            x = blk.forward_nhwc(x)
        x = self.mid_block.forward_nhwc(x)
        n, h, w, c = x.shape
        x = self.conv_norm_out.forward_rows(x.view(n, h * w, c), silu=True).view(n, h, w, c)
        return self.conv_out.forward_nhwc(x)


class Decoder(nn.Module):
    def __init__(self, latent_channels, out_channels, chans: Sequence[int], layers, groups):
        super().__init__()
        rev = list(reversed(chans))
        self.conv_in = LibConv2d(latent_channels, rev[0], 3, padding=1)
        self.mid_block = UNetMidBlock2D(rev[0], groups)
        self.up_blocks = nn.ModuleList()
        c = rev[0]
        for i, co in enumerate(rev):
            self.up_blocks.append(UpDecoderBlock2D(c, co, layers + 1, groups, add_upsample=i < len(rev) - 1))
            c = co
        self.conv_norm_out = GroupNorm(groups, c, eps=1e-6)
        self.conv_act = nn.SiLU()
        self.conv_out = LibConv2d(c, out_channels, 3, padding=1)

    def forward_nhwc(self, z):
        x = self.mid_block.forward_nhwc(self.conv_in.forward_nhwc(z))
        for blk in self.up_blocks:
            x = blk.forward_nhwc(x)
        n, h, w, c = x.shape
        x = self.conv_norm_out.forward_rows(x.view(n, h * w, c), silu=True).view(n, h, w, c)
        return self.conv_out.forward_nhwc(x)


class DiagonalGaussianDistribution:
    """diffusers' posterior object: parameters = cat(mean, logvar) on dim 1, logvar clamped to [-30, 20]."""

    def __init__(self, parameters: torch.Tensor):
        self.mean, logvar = torch.chunk(parameters, 2, dim=1)
        self.logvar = torch.clamp(logvar, -30.0, 20.0)
        self.std = torch.exp(0.5 * self.logvar)

    def sample(self, generator=None) -> torch.Tensor:
        noise = torch.randn(self.mean.shape, generator=generator, device=self.mean.device, dtype=self.mean.dtype)
        return self.mean + self.std * noise

    def mode(self) -> torch.Tensor:
        return self.mean


class AutoencoderKL(nn.Module):
    def __init__(self, in_channels=3, out_channels=3, latent_channels=4, block_out_channels=(128, 256, 512, 512),
                 layers_per_block=2, norm_num_groups=32, scaling_factor=0.18215):
        super().__init__()
        self.encoder = Encoder(in_channels, latent_channels, block_out_channels, layers_per_block, norm_num_groups)
        self.decoder = Decoder(latent_channels, out_channels, block_out_channels, layers_per_block, norm_num_groups)
        self.quant_conv = nn.Conv2d(2 * latent_channels, 2 * latent_channels, 1)
        self.post_quant_conv = nn.Conv2d(latent_channels, latent_channels, 1)
        self.config = SimpleNamespace(scaling_factor=scaling_factor, latent_channels=latent_channels,
                                      block_out_channels=tuple(block_out_channels))

    @property
    def dtype(self):
        return next(self.parameters()).dtype

    def encode(self, x: torch.Tensor):
        """x: [n, 3, H, W] in [-1, 1] -> `.latent_dist` (NCHW tensors, like diffusers)."""
        h = self.encoder.forward_nhwc(to_nhwc(x.to(self.dtype)))
        moments = F.conv2d(to_nchw_view(h), self.quant_conv.weight, self.quant_conv.bias)
        return SimpleNamespace(latent_dist=DiagonalGaussianDistribution(moments))

    def decode(self, z: torch.Tensor):
        """z: [n, 4, h, w] -> `.sample` [n, 3, 8h, 8w]."""
        z = F.conv2d(z.to(self.dtype), self.post_quant_conv.weight, self.post_quant_conv.bias)
        return SimpleNamespace(sample=to_nchw_view(self.decoder.forward_nhwc(to_nhwc(z))))


def decode_latents(vae: AutoencoderKL, latents: torch.Tensor, decode_chunk_size=None) -> torch.Tensor:
    """pipeline_i2vgen_xl.py:443-463 — latents [b, c, f, h, w] -> video [b, 3, f, 8h, 8w] float32.  `decode_chunk_size`
    keeps its meaning (frames per VAE call; None = all at once); the per-frame result does not depend on it."""
    latents = 1 / vae.config.scaling_factor * latents
    b, c, f, h, w = latents.shape
    latents = latents.permute(0, 2, 1, 3, 4).reshape(b * f, c, h, w)
    if decode_chunk_size is not None:
        image = torch.cat([vae.decode(latents[i:i + decode_chunk_size]).sample
                           for i in range(0, latents.shape[0], decode_chunk_size)], dim=0)
    else:
        image = vae.decode(latents).sample
    video = image[None, :].reshape((b, f, -1) + image.shape[2:]).permute(0, 2, 1, 3, 4)
    return video.float()


def encode_vae_video(vae: AutoencoderKL, frames: torch.Tensor, generator=None) -> torch.Tensor:
    """pipeline_i2vgen_xl.py:565-592 after the image pre-processing: frames [f, 3, H, W] in [-1, 1] -> video latents
    [1, c, f, H/8, W/8] (posterior SAMPLE x scaling_factor).  One batched encoder pass; the posterior noise is drawn
    frame by frame in the reference's order so a seeded generator gives the same draws."""
    dist = vae.encode(frames).latent_dist
    lat = []
    for i in range(frames.shape[0]):
        noise = torch.randn(dist.mean[i:i + 1].shape, generator=generator, device=dist.mean.device, dtype=dist.mean.dtype)
        lat.append(((dist.mean[i:i + 1] + dist.std[i:i + 1] * noise) * vae.config.scaling_factor).squeeze(0))
    lat = torch.stack(lat)
    return lat.reshape(1, frames.shape[0], *lat.shape[1:]).permute(0, 2, 1, 3, 4)

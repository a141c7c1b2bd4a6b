"""I2VGen-XL 3-D UNet, B200-native forward.

The module / parameter names are those of diffusers==0.26.3 ``I2VGenXLUNet`` (the model the reference drives at
i2vgen-xl/pipelines/pipeline_i2vgen_xl.py:1146-1155 and whose sub-modules i2vgen-xl/pnp_utils.py patches), so that a
diffusers state_dict loads unchanged and the hook surface (``up_blocks[i].resnets[j]``, ``.attentions[j]
.transformer_blocks[0].attn1.processor``, ``.temp_attentions[j]...``) resolves exactly as in the reference.

What differs is everything underneath:
  * activations are channels-last for the whole network; a frame batch is [B*F, H, W, C] and the same memory viewed
    as [B, F*H*W, C] IS the frame-major token matrix of the temporal layers — the reference's
    [B,C,F,h,w] <-> [B*F,C,h,w] <-> [B*hw,F,C] permute/reshape copies do not exist;
  * GroupNorm+SiLU, every 3x3 conv (implicit GEMM, TMA taps), every temporal (3,1,1) conv, every Linear and all
    self-attention run on the hand-written sm_100a kernels of anyv2v_b200.ops;
  * LayerNorm and the GEGLU gate (fused into the FF GEMM's epilogue) are hand-written too; the few layers SURVEY 8(f)
    leaves as "next" (stride-2 / tiny stem convs, 145-token cross-attention SDPA, nearest up-sampling, skip concat)
    are library calls collected in anyv2v_b200.next_rows.
Public module ``forward``s keep the diffusers protocol (logical NCHW tensors; channels_last memory makes the
conversion a zero-copy view).
"""
from __future__ import annotations

import math
from typing import Optional, Sequence

import torch
import torch.nn as nn

from . import next_rows as nr
from . import ops

I2VGEN_XL_CONFIG = dict(in_channels=4, out_channels=4, block_out_channels=(320, 640, 1280, 1280), layers_per_block=2,
                        norm_num_groups=32, cross_attention_dim=1024, head_dim=64, transformer_in_heads=8)


# ------------------------------------------------------------------------------------------------ layout helpers
def to_nhwc(x: torch.Tensor) -> torch.Tensor:
    """logical [N,C,H,W] -> physical [N,H,W,C] contiguous (zero-copy when x is channels_last)."""
    return x.permute(0, 2, 3, 1).contiguous()


def to_nchw_view(x_nhwc: torch.Tensor) -> torch.Tensor:
    return x_nhwc.permute(0, 3, 1, 2)


class _PackedCache:
    """Re-packed weight (e.g. [Cout][ky][kx][Cin]) cached against the parameter's storage + version counter."""

    def __init__(self):
        self._key = None
        self._val = None

    def get(self, param: torch.Tensor, fn):
        key = (param.data_ptr(), param._version, param.device, param.dtype)
        if key != self._key:
            with torch.no_grad():
                self._val = fn(param).contiguous()
            self._key = key
        return self._val


# ------------------------------------------------------------------------------------------------ leaf layers
class Linear(nn.Linear):
    def forward(self, x, residual=None):
        shp = x.shape
        y = ops.linear(x.reshape(-1, shp[-1]), self.weight, bias=self.bias,
                       residual=None if residual is None else residual.reshape(-1, self.out_features))
        return y.view(*shp[:-1], self.out_features)


class Conv3x3(nn.Conv2d):
    """3x3 / pad 1 convolution run as an implicit GEMM on tcgen05 (ops.conv3x3), stride 1 or 2 (Downsample2D).

    Widths the tensor-core tiles do not cover are padded in the PACKED weight only (the parameter keeps its diffusers shape):
    Cin not a multiple of 64 (conv_in: 8 input channels) -> every tap's K block is zero-padded to 64 and the activation's missing
    channels read as zeros through TMA out-of-bounds fill; Cout not a multiple of 8 (conv_out: 4) -> zero rows up to 8 and the
    caller slices the result."""

    def __init__(self, cin, cout, stride: int = 1):
        super().__init__(cin, cout, 3, stride=stride, padding=1)
        self._packed = _PackedCache()
        self._packed_bias = _PackedCache()
        self.cin_pad = (cin + 63) // 64 * 64
        self.cout_pad = (cout + 7) // 8 * 8

    def packed_weight(self):
        def pack(w):
            co, ci = w.shape[0], w.shape[1]
            wp = w.new_zeros((self.cout_pad, 3, 3, self.cin_pad))
            wp[:co, :, :, :ci] = w.permute(0, 2, 3, 1)
            return wp.reshape(self.cout_pad, -1)
        return self._packed.get(self.weight, pack)

    def packed_bias(self):
        if self.bias is None or self.cout_pad == self.out_channels:
            return self.bias
        return self._packed_bias.get(self.bias, lambda b: torch.cat([b, b.new_zeros(self.cout_pad - b.shape[0])]))

    def forward_nhwc(self, x, rowbias=None, rows_per_rowbias=0, residual=None, out=None, n_slots=1, slot_stride=0):
        y = ops.conv3x3(x, self.packed_weight(), bias=self.packed_bias(), rowbias=rowbias, rows_per_rowbias=rows_per_rowbias,
                        residual=residual, out=out, n_slots=n_slots, slot_stride=slot_stride, stride=self.stride[0])
        return y if self.cout_pad == self.out_channels else y[..., :self.out_channels]

    def forward(self, x):
        return to_nchw_view(self.forward_nhwc(to_nhwc(x)))


class TemporalConv3(nn.Conv3d):
    def __init__(self, dim):
        super().__init__(dim, dim, (3, 1, 1), padding=(1, 0, 0))
        self._packed = _PackedCache()

    def packed_weight(self):
        return self._packed.get(self.weight, lambda w: w[:, :, :, 0, 0].permute(0, 2, 1).reshape(w.shape[0], -1))


class GroupNorm(nn.GroupNorm):
    def forward_rows(self, x_rows: torch.Tensor, silu: bool, x2_rows: Optional[torch.Tensor] = None) -> torch.Tensor:
        """x_rows: [n_samples, rows, C] channels-last; with x2_rows the logical input is [x_rows | x2_rows] along the channels."""
        return ops.groupnorm(x_rows, self.weight, self.bias, self.num_groups, self.eps, silu, x2=x2_rows)


# ------------------------------------------------------------------------------------------------ attention
class AttnProcessor:
    """B200 attention processor with the diffusers protocol (pnp_utils.py:142-150).

    hidden_states is either the protocol's [batch, seq, C] tensor, or — fast path used by this package's temporal
    transformers — a 4-D frame-major view [B, HW, F, C] (strides (F*HW*C, C, HW*C, 1)) so that no transposed copy of
    the tokens is ever made.  ``residual`` (optional, same shape) is added in the out-projection epilogue.
    """

    def inject_now(self) -> bool:
        return False

    def __call__(self, attn, hidden_states, encoder_hidden_states=None, attention_mask=None, temb=None, scale=1.0,
                 residual=None, kv_batch_div: int = 1):
        if attention_mask is not None:
            raise NotImplementedError("attention masks are not used on the I2VGen-XL path")
        if encoder_hidden_states is not None:
            return self._cross(attn, hidden_states, encoder_hidden_states, residual, kv_batch_div)
        return self._self(attn, hidden_states, residual)

    # -- self-attention (spatial: [BF, N, C]; temporal: 4-D frame-major view or [B*HW, F, C])
    def _self(self, attn, x, residual):
        frames_view = x.dim() == 4
        if frames_view:
            B, HW, F, C = x.shape
            assert x.stride() == (F * HW * C, C, HW * C, 1), "expected the frame-major token view"
            tokens = x.permute(0, 2, 1, 3).reshape(B * F * HW, C)  # zero-copy back to the token matrix
            nbatch, seq = B * HW, F
        else:
            nb, seq, C = x.shape
            if seq <= 32 and 128 % seq == 0 and x.is_contiguous():
                # protocol-shaped temporal tokens [B*HW, F, C] (F = 8 / 16 / 32 frames): address them as (pixel, frame);
                # longer short sequences (the 8 x 8 = 64-token spatial attention of the mid block) stay in rows mode, copy-free
                return self._self_protocol_temporal(attn, x, residual)
            tokens = x.reshape(nb * seq, C)
            nbatch = nb
            B = nb
        heads = attn.heads
        rows = tokens.shape[0]
        inject = self.inject_now() and (B % 3 == 0)
        wqkv = attn.fused_qkv_weight()
        out_attn = torch.empty((rows, C), dtype=tokens.dtype, device=tokens.device)
        fusable = frames_view and 128 % seq == 0 and C % 64 == 0 and wqkv.shape[0] == 3 * heads * 64
        if fusable:
            # temporal self-attention: Q/K/V projection fused into the attention kernel (Q, K, V never reach HBM); on injected
            # steps (pnp_utils.py:295-302) Q and K of all three branches are projected from the SOURCE clip inside the kernel
            ops.temporal_attention_fused(tokens, wqkv, heads, seq, HW, B, out_attn, scale=attn.scale, n_v=3 if inject else 1)
        elif not inject:
            qkv = ops.linear(tokens, wqkv)  # [rows, 3C]
            q, k, v = qkv[:, :C], qkv[:, C:2 * C], qkv[:, 2 * C:]
            ops.attention(q, k, v, heads, seq, nbatch, out_attn, scale=attn.scale, frames_mode=frames_view,
                          HW=(HW if frames_view else 0))
        else:
            # PnP injection (pnp_utils.py:189-196): q,k of the uncond/cond chunks == the source chunk's, so only the
            # source third is projected to q,k and the probabilities are shared by the three V branches.
            src_rows = rows // 3
            qk = ops.linear(tokens[:src_rows], wqkv[:2 * C])          # [rows/3, 2C]
            v = ops.linear(tokens, wqkv[2 * C:])                      # [rows, C]
            ops.attention(qk[:, :C], qk[:, C:], v, heads, seq, nbatch // 3, out_attn, scale=attn.scale, n_v=3,
                          v_branch_stride=src_rows * C, o_branch_stride=src_rows * C, frames_mode=frames_view,
                          HW=(HW if frames_view else 0))
        res2d = None
        if residual is not None:
            res2d = residual.permute(0, 2, 1, 3).reshape(rows, C) if frames_view else residual.reshape(rows, C)
        y = ops.linear(out_attn, attn.to_out[0].weight, bias=attn.to_out[0].bias, residual=res2d)
        if frames_view:
            return y.view(B, F, HW, C).permute(0, 2, 1, 3)
        return y.view(x.shape)

    def _self_protocol_temporal(self, attn, x, residual):
        # [B*HW, F, C] contiguous: make it frame-major once (copy), run the fast path, convert back.
        nb, F, C = x.shape
        xt = x.transpose(0, 1).contiguous().view(1, F, nb, C).permute(0, 2, 1, 3)  # [1, nb, F, C] frame-major view
        rt = None
        if residual is not None:
            rt = residual.transpose(0, 1).contiguous().view(1, F, nb, C).permute(0, 2, 1, 3)
        if self.inject_now() and nb % 3 == 0:
            # keep branch-major grouping: [3, nb/3, F, C]
            xt = x.view(3, nb // 3, F, C).transpose(1, 2).contiguous().permute(0, 2, 1, 3)
            if residual is not None:
                rt = residual.view(3, nb // 3, F, C).transpose(1, 2).contiguous().permute(0, 2, 1, 3)
        y = self._self(attn, xt, rt)  # [B', HW', F, C] view over frame-major memory
        return y.reshape(nb, F, C).contiguous()  # back to the protocol layout [nb][F][C] (copy; short sequences only)

    def _cross(self, attn, x, ctx, residual, kv_div: int = 1):
        """Cross-attention to the 145-token context.  ``ctx`` may hold ONE context per clip ([nb/kv_div, Nk, D]): the
        reference repeat_interleaves it over the frames and projects K/V per frame; here K/V are projected once per
        clip and the kernel maps query sequence b to key/value sequence b // kv_div."""
        nb, seq, C = x.shape
        nk = ctx.shape[1]
        assert ctx.shape[0] * kv_div == nb
        q = ops.linear(x.reshape(nb * seq, C), attn.to_q.weight)
        kv = ops.linear(ctx.reshape(-1, ctx.shape[-1]), attn.fused_kv_weight())      # [nb/kv_div * Nk, 2C]
        o = torch.empty((nb * seq, C), dtype=x.dtype, device=x.device)
        ops.attention(q, kv[:, :C], kv[:, C:], attn.heads, seq, nb, o, scale=attn.scale, seq_kv=nk, kv_batch_div=kv_div)
        y = ops.linear(o, attn.to_out[0].weight, bias=attn.to_out[0].bias,
                       residual=None if residual is None else residual.reshape(nb * seq, C))
        return y.view(nb, seq, C)


class Attention(nn.Module):
    """diffusers ``Attention`` attribute surface (consisti2v/.../videoldm_attention.py:64-177): q/k/v without bias,
    to_out = [Linear(bias), Dropout], dispatch through the instance attribute ``processor``."""

    def __init__(self, query_dim, cross_attention_dim=None, heads=8, dim_head=64):
        super().__init__()
        inner = heads * dim_head
        self.heads = heads
        self.scale = dim_head ** -0.5
        self.spatial_norm = None
        self.group_norm = None
        self.norm_cross = None
        self.residual_connection = False
        self.rescale_output_factor = 1.0
        self.to_q = nn.Linear(query_dim, inner, bias=False)
        self.to_k = nn.Linear(cross_attention_dim or query_dim, inner, bias=False)
        self.to_v = nn.Linear(cross_attention_dim or query_dim, inner, bias=False)
        self.to_out = nn.ModuleList([nn.Linear(inner, query_dim, bias=True), nn.Dropout(0.0)])
        self.processor = AttnProcessor()
        self._qkv = _PackedCache()
        self._kv = _PackedCache()

    def fused_qkv_weight(self):
        key_param = self.to_q.weight
        val = self._qkv.get(key_param, lambda w: torch.cat([w, self.to_k.weight, self.to_v.weight], dim=0))
        return val

    def fused_kv_weight(self):
        return self._kv.get(self.to_k.weight, lambda w: torch.cat([w, self.to_v.weight], dim=0))

    def prepare_attention_mask(self, *a, **k):
        raise NotImplementedError("attention masks are not used on the I2VGen-XL path")

    def forward(self, hidden_states, encoder_hidden_states=None, attention_mask=None, **kw):
        return self.processor(self, hidden_states, encoder_hidden_states=encoder_hidden_states,
                              attention_mask=attention_mask, **kw)


class _GEGLU(nn.Module):
    def __init__(self, dim_in, dim_out):
        super().__init__()
        self.proj = Linear(dim_in, dim_out * 2)
        self._packed = _PackedCache()

    def packed(self):
        """(weight, bias) with the h / gate halves interleaved in blocks of 32 rows: the layout of the fused GEGLU
        epilogue (csrc/gemm_tcgen05.cu), which stores h * gelu_erf(gate) and never materialises the [rows, 8C] tensor."""
        w = self.proj.weight
        key = (w.data_ptr(), w._version, self.proj.bias.data_ptr(), self.proj.bias._version)
        if self._packed._key != key:
            with torch.no_grad():
                self._packed._val = ops.geglu_pack(w, self.proj.bias)
            self._packed._key = key
        return self._packed._val


class _GELU(nn.Module):
    def __init__(self, dim_in, dim_out):
        super().__init__()
        self.proj = nn.Linear(dim_in, dim_out)


class FeedForward(nn.Module):
    def __init__(self, dim, activation_fn="geglu", inner_dim=None):
        super().__init__()
        inner = inner_dim or dim * 4
        self.geglu = activation_fn == "geglu"
        act = _GEGLU(dim, inner) if self.geglu else _GELU(dim, inner)
        self.net = nn.ModuleList([act, nn.Dropout(0.0), Linear(inner, dim) if self.geglu else nn.Linear(inner, dim)])

    def forward(self, x, residual=None):
        if self.geglu:
            wp, bp = self.net[0].packed()
            shp = x.shape
            h = ops.linear(x.reshape(-1, shp[-1]), wp, bias=bp, geglu=True).view(*shp[:-1], wp.shape[0] // 2)
            return self.net[2](h, residual=residual)
        h = torch.nn.functional.gelu(torch.nn.functional.linear(x, self.net[0].proj.weight, self.net[0].proj.bias))
        y = torch.nn.functional.linear(h, self.net[2].weight, self.net[2].bias)
        return y if residual is None else y + residual


class BasicTransformerBlock(nn.Module):
    """LN -> attn1 -> + ; LN -> attn2 -> + ; LN -> GEGLU FF -> +  (videoldm_transformer_blocks.py:461-562).
    Residual adds are fused into the producing GEMM's epilogue."""

    def __init__(self, dim, heads, head_dim, cross_attention_dim=None, double_self_attention=False):
        super().__init__()
        self.norm1 = nn.LayerNorm(dim, eps=1e-5)
        self.attn1 = Attention(dim, None, heads, head_dim)
        self.norm2 = nn.LayerNorm(dim, eps=1e-5)
        self.attn2 = Attention(dim, None if double_self_attention else cross_attention_dim, heads, head_dim)
        self.norm3 = nn.LayerNorm(dim, eps=1e-5)
        self.ff = FeedForward(dim)

    @staticmethod
    def _ln(norm, x):
        return ops.layernorm(x, norm.weight, norm.bias, norm.eps)

    def forward(self, x, encoder_hidden_states=None, kv_batch_div: int = 1, expand=None):
        """x: [batch, seq, C], or the 4-D frame-major view [B, HW, F, C] (whose base memory is [B, F, HW, C]).
        Row-wise layers (LayerNorm, FF) always run on the contiguous base; only attention sees the view.
        ``expand``: a map applied to the hidden states right after attn1 — duplication of the shared edit branch
        (shared-prefix mode of I2VGenXLUNet.forward: the last point at which uncond and cond are still identical) or
        removal of the source branch after its last live site (_SourcePrune)."""
        frames_view = x.dim() == 4
        flip = (lambda t: t.permute(0, 2, 1, 3)) if frames_view else (lambda t: t)
        base = flip(x)  # contiguous
        base = flip(self.attn1(flip(self._ln(self.norm1, base)), encoder_hidden_states=None, residual=flip(base)))
        if expand is not None:
            base = expand(base)  # leading dim of the contiguous base = frames (spatial) or clips (temporal)
        kw = {"kv_batch_div": kv_batch_div} if encoder_hidden_states is not None and kv_batch_div != 1 else {}
        base = flip(self.attn2(flip(self._ln(self.norm2, base)), encoder_hidden_states=encoder_hidden_states,
                               residual=flip(base), **kw))
        base = self.ff(self._ln(self.norm3, base), residual=base)
        return flip(base)


class Transformer2DModel(nn.Module):
    def __init__(self, heads, head_dim, in_channels, cross_attention_dim, groups=32):
        super().__init__()
        inner = heads * head_dim
        self.norm = GroupNorm(groups, in_channels, eps=1e-6)
        self.proj_in = Linear(in_channels, inner)
        self.transformer_blocks = nn.ModuleList([BasicTransformerBlock(inner, heads, head_dim, cross_attention_dim)])
        self.proj_out = Linear(inner, in_channels)

    def forward_nhwc(self, x, ctx, expand=None):
        """ctx: [NF, Nk, D] (diffusers protocol) or one context per clip [B, Nk, D] with NF % B == 0.
        ``expand``: see BasicTransformerBlock.forward — x then holds the UNIQUE branches only and the result all of them."""
        nf, h, w, c = x.shape
        y = self.norm.forward_rows(x.view(nf, h * w, c), silu=False)
        y = self.proj_in(y)
        res = x.view(nf, h * w, c)
        if expand is not None:
            assert len(self.transformer_blocks) == 1
            res = expand(res)
            nf = res.shape[0]
        for blk in self.transformer_blocks:
            y = blk(y, encoder_hidden_states=ctx, kv_batch_div=nf // ctx.shape[0], expand=expand)
        return self.proj_out(y, residual=res).view(nf, h, w, c)

    def forward(self, hidden_states, encoder_hidden_states=None, **kw):
        return (to_nchw_view(self.forward_nhwc(to_nhwc(hidden_states), encoder_hidden_states)),)


class TransformerTemporalModel(nn.Module):
    def __init__(self, heads, head_dim, in_channels, groups=32):
        super().__init__()
        inner = heads * head_dim
        self.norm = GroupNorm(groups, in_channels, eps=1e-6)
        self.proj_in = Linear(in_channels, inner)
        self.transformer_blocks = nn.ModuleList([BasicTransformerBlock(inner, heads, head_dim, None, True)])
        self.proj_out = Linear(inner, in_channels)

    def forward_nhwc(self, x, num_frames, expand=None):
        bf, h, w, c = x.shape
        b, f, hw = bf // num_frames, num_frames, h * w
        y = self.norm.forward_rows(x.view(b, f * hw, c), silu=False)        # per-clip statistics
        y = self.proj_in(y)                                                 # [b, f*hw, inner] frame-major tokens
        inner = y.shape[-1]
        y4 = y.view(b, f, hw, inner).permute(0, 2, 1, 3)                    # [b, hw, f, inner] view, no copy
        res = x.view(b, f * hw, c)
        if expand is not None:                                              # clips are dropped right after attn1
            assert len(self.transformer_blocks) == 1
            res = expand(res)
            b = res.shape[0]
        for blk in self.transformer_blocks:
            y4 = blk(y4, encoder_hidden_states=None, expand=expand)
        y = y4.permute(0, 2, 1, 3).reshape(b, f * hw, inner)
        return self.proj_out(y, residual=res).view(b * f, h, w, c)

    def forward(self, hidden_states, num_frames=1, **kw):
        return (to_nchw_view(self.forward_nhwc(to_nhwc(hidden_states), num_frames)),)


# ------------------------------------------------------------------------------------------------ conv blocks
class _Temb:
    """The time embedding of a step together with its SiLU: every resnet applies ``time_emb_proj(SiLU(temb))`` (pnp_utils.py:89-91)
    to the SAME temb, so the activation is computed once per step instead of once per resnet.  Slices like a tensor."""
    __slots__ = ("raw", "act")

    def __init__(self, raw, act=None):
        self.raw = raw
        self.act = nr.silu(raw) if act is None else act

    def __getitem__(self, sl):
        return _Temb(self.raw[sl], self.act[sl])

    @property
    def shape(self):
        return self.raw.shape


class ResnetBlock2D(nn.Module):
    """GN -> SiLU -> conv1 (+temb in the epilogue) -> GN -> SiLU -> conv2 (+shortcut in the epilogue)
    (pnp_utils.py:41-126 is the reference's full restatement of this block)."""

    def __init__(self, in_channels, out_channels, temb_channels, groups=32, eps=1e-5):
        super().__init__()
        self.in_channels, self.out_channels = in_channels, out_channels
        self.norm1 = GroupNorm(groups, in_channels, eps=eps)
        self.conv1 = Conv3x3(in_channels, out_channels)
        self.time_emb_proj = Linear(temb_channels, out_channels)
        self.norm2 = GroupNorm(groups, out_channels, eps=eps)
        self.dropout = nn.Dropout(0.0)
        self.conv2 = Conv3x3(out_channels, out_channels)
        self.nonlinearity = nn.SiLU()
        self.upsample = None
        self.downsample = None
        self.skip_time_act = False
        self.time_embedding_norm = "default"
        self.output_scale_factor = 1.0
        self.conv_shortcut = nn.Conv2d(in_channels, out_channels, 1) if in_channels != out_channels else None

    def shortcut_nhwc(self, x, skip=None):
        if self.conv_shortcut is None:
            return x
        nf, h, w, c1 = x.shape
        cin = self.in_channels
        w2 = self.conv_shortcut.weight.view(self.out_channels, cin)
        a2 = None if skip is None else skip.view(-1, cin - c1)
        return ops.linear(x.view(-1, c1), w2, bias=self.conv_shortcut.bias, a2=a2).view(nf, h, w, self.out_channels)

    def forward_nhwc(self, x, temb, inject: bool = False, skip=None, temb_act=None):
        """``skip`` (up blocks): the block's input is the channel concat [x | skip] (diffusers: torch.cat([hidden_states,
        res_hidden_states], dim=1)); it is never materialised — GroupNorm reads the two sources and writes the normalised
        concat, the 1x1 shortcut runs its K loop over both.  ``temb_act`` = SiLU(temb), computed once per step by the caller."""
        nf, h, w, c1 = x.shape
        cin = self.in_channels
        hw = h * w
        if skip is not None and (c1 % 64 != 0 or inject):
            x, skip = torch.cat([x, skip], dim=-1), None   # widths the two-source K loop does not cover / the injected resnet
            c1 = cin
        if isinstance(temb, _Temb):
            temb, temb_act = temb.raw, temb.act
        tproj = self.time_emb_proj(nr.silu(temb) if temb_act is None else temb_act)   # [NF, Cout]
        short = self.shortcut_nhwc(x, skip)
        if not inject:
            y = self.norm1.forward_rows(x.view(nf, hw, c1), silu=True, x2_rows=None if skip is None else skip.view(nf, hw, cin - c1))
            y = y.view(nf, h, w, cin)
            y = self.conv1.forward_nhwc(y, rowbias=tproj, rows_per_rowbias=hw)
            y = self.norm2.forward_rows(y.view(nf, hw, -1), silu=True).view(nf, h, w, -1)
            return self.conv2.forward_nhwc(y, residual=short)
        # PnP feature injection (pnp_utils.py:109-115): h[uncond] = h[cond] = h[source].  Only the source third of
        # norm1/conv1/norm2/conv2 is live; conv2's epilogue writes the shared tile to the three branch slots, each
        # with its own shortcut — the injection copy is the store itself.
        n = nf // 3
        xs = x[:n]
        y = self.norm1.forward_rows(xs.reshape(n, hw, cin), silu=True).view(n, h, w, cin)
        y = self.conv1.forward_nhwc(y, rowbias=tproj[:n], rows_per_rowbias=hw)
        y = self.norm2.forward_rows(y.view(n, hw, -1), silu=True).view(n, h, w, -1)
        out = torch.empty((nf, h, w, self.out_channels), dtype=x.dtype, device=x.device)
        self.conv2.forward_nhwc(y, residual=short, out=out, n_slots=3, slot_stride=n * hw * self.out_channels)
        return out

    def forward(self, input_tensor, temb, scale: float = 1.0):
        return to_nchw_view(self.forward_nhwc(to_nhwc(input_tensor), temb))


class TemporalConvLayer(nn.Module):
    def __init__(self, dim, groups=32, dropout=0.1):
        super().__init__()
        self.conv1 = nn.Sequential(GroupNorm(groups, dim), nn.SiLU(), TemporalConv3(dim))
        for name in ("conv2", "conv3", "conv4"):
            setattr(self, name, nn.Sequential(GroupNorm(groups, dim), nn.SiLU(), nn.Dropout(dropout), TemporalConv3(dim)))
        nn.init.zeros_(self.conv4[-1].weight)
        nn.init.zeros_(self.conv4[-1].bias)

    def forward_nhwc(self, x, num_frames):
        bf, h, w, c = x.shape
        b, hw = bf // num_frames, h * w
        ident = x.view(b, num_frames * hw, c)
        y = ident
        for i, seq in enumerate((self.conv1, self.conv2, self.conv3, self.conv4)):
            y = seq[0].forward_rows(y, silu=True)
            conv = seq[-1]
            y = ops.tconv3(y, conv.packed_weight(), num_frames, hw, bias=conv.bias, residual=ident if i == 3 else None)
        return y.view(bf, h, w, c)

    def forward(self, hidden_states, num_frames=1):
        return to_nchw_view(self.forward_nhwc(to_nhwc(hidden_states), num_frames))


class Downsample2D(nn.Module):
    def __init__(self, channels):
        super().__init__()
        self.conv = Conv3x3(channels, channels, stride=2)

    def forward_nhwc(self, x):
        return self.conv.forward_nhwc(x)

    def forward(self, x, scale: float = 1.0):
        return to_nchw_view(self.forward_nhwc(to_nhwc(x)))


class Upsample2D(nn.Module):
    """nearest-neighbour x 2, then conv 3 x 3 (diffusers Upsample2D(use_conv=True); twin at seine/models/resnet.py:24-76) — computed
    straight from the low-resolution input: each of the four output phases (2i+py, 2j+px) is a 2 x 2 convolution with pre-summed
    taps (ops.upsample2x_conv3x3), so the 4x larger up-sampled tensor is never written or read and the layer costs 4/9 of its
    FLOPs.  The parameter keeps its diffusers shape [C, C, 3, 3]; the phase weights are a cached re-packing."""

    def __init__(self, channels):
        super().__init__()
        self.conv = Conv3x3(channels, channels)
        self._phases = _PackedCache()

    def phase_weights(self):
        return self._phases.get(self.conv.weight, ops.pack_upsample_weights)

    def forward_nhwc(self, x):
        return ops.upsample2x_conv3x3(x, self.phase_weights(), bias=self.conv.bias)

    def forward(self, x, output_size=None, scale: float = 1.0):
        return to_nchw_view(self.forward_nhwc(to_nhwc(x)))


class _SourcePrune:
    """Round-2 candidate (AV2V_PRUNE_SOURCE, set by the PnP edit loop): the source branch's noise prediction is discarded
    (pipeline :1160), so the branch is dead after its LAST firing injection site of the step (SURVEY 8a iii).  `site` =
    (up block, layer, "resnet" | "spatial" | "temporal"); from there on the batch holds the edit branches only."""

    def __init__(self, site, frames: int):
        self.site, self.f, self.done = tuple(site), int(frames), False

    def frames(self, t):   # [B*F, ...] -> [(B-1)*F, ...]
        return t[self.f:]

    def clips(self, t):    # [B, ...] -> [B-1, ...]
        return t[1:]

    def at(self, block, layer, kind) -> bool:
        return (not self.done) and self.site == (block, layer, kind)


class _Block3D(nn.Module):
    def _layer(self, i, x, temb, ctx, nframes, prune=None, block_index=None, skip=None):
        """-> (x, temb, ctx); temb / ctx come back shortened when `prune` dropped the source branch inside this layer.
        ``skip`` (up blocks): the resnet's input is the channel concat [x | skip], materialised only for a patched resnet."""
        res = self.resnets[i]
        # instance-level forward overrides (register_conv_injection) follow the NCHW protocol of the reference (one tensor)
        if "forward" in res.__dict__:
            if skip is not None:
                x = torch.cat([x, skip], dim=-1)
            x = to_nhwc(res(to_nchw_view(x), temb.raw if isinstance(temb, _Temb) else temb))
        else:
            x = res.forward_nhwc(x, temb, skip=skip)
        if prune is not None and prune.at(block_index, i, "resnet"):
            x, temb, ctx, prune.done = prune.frames(x), prune.frames(temb), prune.clips(ctx), True
        x = self.temp_convs[i].forward_nhwc(x, nframes)
        if self.has_cross_attention:
            if prune is not None and prune.at(block_index, i, "spatial"):
                temb, ctx, prune.done = prune.frames(temb), prune.clips(ctx), True
                x = self.attentions[i].forward_nhwc(x, ctx, expand=prune.frames)   # attn1 on all branches, the rest on the edit ones
            else:
                x = self.attentions[i].forward_nhwc(x, ctx)
            if prune is not None and prune.at(block_index, i, "temporal"):
                temb, ctx, prune.done = prune.frames(temb), prune.clips(ctx), True
                x = self.temp_attentions[i].forward_nhwc(x, nframes, expand=prune.clips)
            else:
                x = self.temp_attentions[i].forward_nhwc(x, nframes)
        return x, temb, ctx


class DownBlock3D(_Block3D):
    def __init__(self, in_ch, out_ch, temb_ch, layers, hd, cross_dim, groups, attn, add_downsample):
        super().__init__()
        self.has_cross_attention = attn
        self.resnets = nn.ModuleList(ResnetBlock2D(in_ch if i == 0 else out_ch, out_ch, temb_ch, groups) for i in range(layers))
        self.temp_convs = nn.ModuleList(TemporalConvLayer(out_ch, groups) for _ in range(layers))
        if attn:
            self.attentions = nn.ModuleList(Transformer2DModel(out_ch // hd, hd, out_ch, cross_dim, groups) for _ in range(layers))
            self.temp_attentions = nn.ModuleList(TransformerTemporalModel(out_ch // hd, hd, out_ch, groups) for _ in range(layers))
        self.downsamplers = nn.ModuleList([Downsample2D(out_ch)]) if add_downsample else None

    def forward_nhwc(self, x, temb, ctx, nframes, first_layer: int = 0):
        outs = []
        for i in range(first_layer, len(self.resnets)):
            x, _, _ = self._layer(i, x, temb, ctx, nframes)
            outs.append(x)
        if self.downsamplers is not None:
            x = self.downsamplers[0].forward_nhwc(x)
            outs.append(x)
        return x, outs


class UpBlock3D(_Block3D):
    def __init__(self, in_ch, out_ch, prev_ch, temb_ch, layers, hd, cross_dim, groups, attn, add_upsample):
        super().__init__()
        self.has_cross_attention = attn
        self.resnets = nn.ModuleList(
            ResnetBlock2D((prev_ch if i == 0 else out_ch) + (in_ch if i == layers - 1 else out_ch), out_ch, temb_ch, groups)
            for i in range(layers))
        self.temp_convs = nn.ModuleList(TemporalConvLayer(out_ch, groups) for _ in range(layers))
        if attn:
            self.attentions = nn.ModuleList(Transformer2DModel(out_ch // hd, hd, out_ch, cross_dim, groups) for _ in range(layers))
            self.temp_attentions = nn.ModuleList(TransformerTemporalModel(out_ch // hd, hd, out_ch, groups) for _ in range(layers))
        self.upsamplers = nn.ModuleList([Upsample2D(out_ch)]) if add_upsample else None

    def forward_nhwc(self, x, skips, temb, ctx, nframes, prune=None, block_index=None):
        for i in range(len(self.resnets)):
            skip = skips.pop()
            if skip.shape[0] != x.shape[0]:       # the source branch was pruned: keep the edit branches' frames
                skip = skip[skip.shape[0] - x.shape[0]:]
            x, temb, ctx = self._layer(i, x, temb, ctx, nframes, prune, block_index, skip=skip)
        if self.upsamplers is not None:
            x = self.upsamplers[0].forward_nhwc(x)
        return x


class MidBlock3D(nn.Module):
    def __init__(self, ch, temb_ch, hd, cross_dim, groups):
        super().__init__()
        self.resnets = nn.ModuleList([ResnetBlock2D(ch, ch, temb_ch, groups), ResnetBlock2D(ch, ch, temb_ch, groups)])
        self.temp_convs = nn.ModuleList([TemporalConvLayer(ch, groups), TemporalConvLayer(ch, groups)])
        self.attentions = nn.ModuleList([Transformer2DModel(ch // hd, hd, ch, cross_dim, groups)])
        self.temp_attentions = nn.ModuleList([TransformerTemporalModel(ch // hd, hd, ch, groups)])

    def forward_nhwc(self, x, temb, ctx, nframes):
        x = self.temp_convs[0].forward_nhwc(self.resnets[0].forward_nhwc(x, temb), nframes)
        x = self.attentions[0].forward_nhwc(x, ctx)
        x = self.temp_attentions[0].forward_nhwc(x, nframes)
        return self.temp_convs[1].forward_nhwc(self.resnets[1].forward_nhwc(x, temb), nframes)


# ------------------------------------------------------------------------------------------------ embeddings / stem
def timestep_embedding(t: torch.Tensor, dim: int) -> torch.Tensor:
    half = dim // 2
    freq = torch.exp(-math.log(10000.0) * torch.arange(half, dtype=torch.float32, device=t.device) / half)
    arg = t[:, None].float() * freq[None, :]
    return torch.cat([torch.cos(arg), torch.sin(arg)], dim=-1)  # flip_sin_to_cos=True


class TimestepEmbedding(nn.Module):
    def __init__(self, in_ch, dim):
        super().__init__()
        self.linear_1 = Linear(in_ch, dim)
        self.act = nn.SiLU()
        self.linear_2 = Linear(dim, dim)

    def forward(self, x):
        return self.linear_2(nr.silu(self.linear_1(x)))


class I2VGenXLTransformerTemporalEncoder(nn.Module):
    """LayerNorm(4) -> 2-head x dim-4 self-attention -> + ; GELU FF(16) -> +  on [B*h*w, F, 4] (tiny: library ops)."""

    def __init__(self, dim, heads, head_dim, ff_inner_dim):
        super().__init__()
        self.norm1 = nn.LayerNorm(dim, eps=1e-5)
        self.attn1 = Attention(dim, None, heads, head_dim)
        self.ff = FeedForward(dim, activation_fn="gelu", inner_dim=ff_inner_dim)

    def forward(self, x):
        F_ = torch.nn.functional
        n = nr.layer_norm(x, self.norm1.weight, self.norm1.bias, 1e-5)
        a = self.attn1
        o = nr.tiny_self_attention(F_.linear(n, a.to_q.weight), F_.linear(n, a.to_k.weight), F_.linear(n, a.to_v.weight), a.heads)
        x = F_.linear(o, a.to_out[0].weight, a.to_out[0].bias) + x
        return self.ff(x, residual=x)


class I2VGenXLUNet(nn.Module):
    def __init__(self, in_channels=4, out_channels=4, block_out_channels: Sequence[int] = (320, 640, 1280, 1280),
                 layers_per_block=2, norm_num_groups=32, cross_attention_dim=1024, head_dim=64, transformer_in_heads=8):
        super().__init__()
        self.config = dict(in_channels=in_channels, out_channels=out_channels, block_out_channels=tuple(block_out_channels),
                           layers_per_block=layers_per_block, norm_num_groups=norm_num_groups,
                           cross_attention_dim=cross_attention_dim, head_dim=head_dim,
                           transformer_in_heads=transformer_in_heads)
        c0, g, temb = block_out_channels[0], norm_num_groups, block_out_channels[0] * 4
        cin = in_channels
        self.conv_in = Conv3x3(cin * 2, c0)
        self.transformer_in = TransformerTemporalModel(transformer_in_heads, head_dim, c0, g)
        self.image_latents_proj_in = nn.Sequential(nn.Conv2d(4, cin * 4, 3, padding=1), nn.SiLU(),
                                                   nn.Conv2d(cin * 4, cin * 4, 3, padding=1), nn.SiLU(),
                                                   nn.Conv2d(cin * 4, cin, 3, padding=1))
        self.image_latents_temporal_encoder = I2VGenXLTransformerTemporalEncoder(cin, 2, cin, cin * 4)
        self.image_latents_context_embedding = nn.Sequential(
            nn.Conv2d(4, cin * 8, 3, padding=1), nn.SiLU(), nn.AdaptiveAvgPool2d((32, 32)),
            nn.Conv2d(cin * 8, cin * 16, 3, stride=2, padding=1), nn.SiLU(),
            nn.Conv2d(cin * 16, cross_attention_dim, 3, stride=2, padding=1))
        self.time_embedding = TimestepEmbedding(c0, temb)
        self.context_embedding = nn.Sequential(Linear(cross_attention_dim, temb), nn.SiLU(),
                                               Linear(temb, cross_attention_dim * cin))
        self.fps_embedding = nn.Sequential(Linear(c0, temb), nn.SiLU(), Linear(temb, temb))
        n = len(block_out_channels)
        self.down_blocks = nn.ModuleList()
        out_ch = c0
        for i, ch in enumerate(block_out_channels):
            in_ch, out_ch = out_ch, ch
            self.down_blocks.append(DownBlock3D(in_ch, out_ch, temb, layers_per_block, head_dim, cross_attention_dim, g,
                                                attn=i < n - 1, add_downsample=i < n - 1))
        self.mid_block = MidBlock3D(block_out_channels[-1], temb, head_dim, cross_attention_dim, g)
        self.up_blocks = nn.ModuleList()
        rev = list(reversed(block_out_channels))
        out_ch = rev[0]
        for i in range(n):
            prev, out_ch = out_ch, rev[i]
            self.up_blocks.append(UpBlock3D(rev[min(i + 1, n - 1)], out_ch, prev, temb, layers_per_block + 1, head_dim,
                                            cross_attention_dim, g, attn=i > 0, add_upsample=i < n - 1))
        self.conv_norm_out = GroupNorm(g, c0, eps=1e-5)
        self.conv_act = nn.SiLU()
        self.conv_out = Conv3x3(c0, out_channels)

    @property
    def dtype(self):
        return self.conv_in.weight.dtype

    # -- conditioning that does not depend on the timestep or the latents: computed once per clip, not per step
    @torch.no_grad()
    def precompute_conditioning(self, fps, image_latents, image_embeddings, encoder_hidden_states):
        b, c, f, h, w = image_latents.shape
        dt = self.dtype
        c0 = self.config["block_out_channels"][0]
        fps_emb = self.fps_embedding(timestep_embedding(fps.reshape(-1).expand(b), c0).to(dt))
        lat_ctx = self.image_latents_context_embedding(image_latents[:, :, 0])
        lat_ctx = lat_ctx.permute(0, 2, 3, 1).reshape(b, -1, lat_ctx.shape[1])
        img_ctx = self.context_embedding(image_embeddings).view(-1, self.config["in_channels"], self.config["cross_attention_dim"])
        # one 145-token context per clip: the reference repeat_interleaves it over the frames (and re-projects K/V for
        # every frame); the attention kernel instead maps frame b*F+f to context b (kv_batch_div = F)
        ctx = torch.cat([encoder_hidden_states, lat_ctx, img_ctx], dim=1).contiguous()
        il = image_latents.permute(0, 2, 1, 3, 4).reshape(b * f, c, h, w)
        il = self.image_latents_proj_in(il)
        il = il[None, :].reshape(b, f, c, h, w).permute(0, 3, 4, 1, 2).reshape(b * h * w, f, c)
        il = self.image_latents_temporal_encoder(il)
        il = il.reshape(b, h, w, f, c).permute(0, 3, 1, 2, 4).reshape(b * f, h, w, c).contiguous()  # NHWC frames
        return dict(fps_emb=fps_emb, ctx=ctx, image_latents_nhwc=il)

    def forward(self, sample, timestep, fps=None, image_latents=None, image_embeddings=None,
                encoder_hidden_states=None, cross_attention_kwargs=None, return_dict: bool = False, cond=None,
                shared_edit_prefix: bool = False, prune_source_after=None):
        """Same call as pipeline_i2vgen_xl.py:1146-1155.  ``cond`` (optional) is precompute_conditioning()'s result.

        ``shared_edit_prefix`` (round-2 candidate, set by the PnP edit loop only): the caller guarantees that the LAST TWO
        branches of the batch — uncond and cond of pipeline :1136 — have the same latents, image latents, fps and
        timestep.  They then differ only through the context of the cross-attentions, so everything up to (and including)
        the first self-attention of down_blocks[0].attentions[0] — conv_in, transformer_in, resnets[0], temp_convs[0],
        GroupNorm / proj_in / attn1 of the first spatial transformer — is computed ONCE for the pair and duplicated right
        before the first cross-attention.  Same results (every normalisation is per sample), ~1/3 less work there.

        ``prune_source_after`` (round-2 candidate, set by the PnP edit loop only): (up block, layer, "resnet" | "spatial" |
        "temporal") of the LAST injection site that fires in this step; the source branch (branch 0) is dropped right after
        it and the result holds the remaining branches only ([uncond, cond])."""
        b, c, f, h, w = sample.shape
        dt = self.dtype
        if cond is None:
            cond = self.precompute_conditioning(fps, image_latents, image_embeddings, encoder_hidden_states)
        t = timestep if torch.is_tensor(timestep) else torch.tensor([timestep], device=sample.device)
        t = t.reshape(-1).to(sample.device).expand(b)
        c0 = self.config["block_out_channels"][0]
        emb = self.time_embedding(timestep_embedding(t, c0).to(dt)) + cond["fps_emb"]
        emb = _Temb(emb.repeat_interleave(f, dim=0).contiguous())                           # [B*F, 4*c0] (+ its SiLU, once per step)
        blk0 = self.down_blocks[0]
        shared = (bool(shared_edit_prefix) and b >= 2 and blk0.has_cross_attention
                  and "forward" not in blk0.resnets[0].__dict__)
        u = b - 1 if shared else b                                                          # unique branches in the prefix
        x = sample[:u].permute(0, 2, 3, 4, 1).reshape(u * f, h, w, c)                       # NHWC frames
        x = torch.cat([x, cond["image_latents_nhwc"][:u * f]], dim=-1)
        x = self.conv_in.forward_nhwc(x)
        x = self.transformer_in.forward_nhwc(x, f)
        if not shared:
            skips = [x]
            down_rest = self.down_blocks
        else:
            expand = lambda t_: torch.cat([t_, t_[-f:]], dim=0)                             # [u*F, ...] -> [b*F, ...]
            skips = [expand(x)]
            x = blk0.resnets[0].forward_nhwc(x, emb[:u * f])
            x = blk0.temp_convs[0].forward_nhwc(x, f)
            x = blk0.attentions[0].forward_nhwc(x, cond["ctx"], expand=expand)              # all b branches from here on
            x = blk0.temp_attentions[0].forward_nhwc(x, f)
            skips.append(x)
            x, outs = blk0.forward_nhwc(x, emb, cond["ctx"], f, first_layer=1)
            skips.extend(outs)
            down_rest = list(self.down_blocks)[1:]
        for blk in down_rest:
            x, outs = blk.forward_nhwc(x, emb, cond["ctx"], f)
            skips.extend(outs)
        x = self.mid_block.forward_nhwc(x, emb, cond["ctx"], f)
        prune = _SourcePrune(prune_source_after, f) if (prune_source_after is not None and b >= 2) else None
        ctx = cond["ctx"]
        for bi, blk in enumerate(self.up_blocks):
            x = blk.forward_nhwc(x, skips, emb, ctx, f, prune, bi)
            if prune is not None and prune.done and emb.shape[0] != x.shape[0]:
                emb, ctx = prune.frames(emb), prune.clips(ctx)
        if prune is not None:
            assert prune.done, f"prune site {prune.site} was never reached"
            b = b - 1
        nf = b * f
        x = self.conv_norm_out.forward_rows(x.view(nf, h * w, -1), silu=True).view(nf, h, w, -1)
        x = self.conv_out.forward_nhwc(x)                                                    # [B*F, h, w, 4]
        out = x.view(b, f, h, w, -1).permute(0, 4, 1, 2, 3).contiguous()                     # [B, 4, F, h, w]
        return (out,)

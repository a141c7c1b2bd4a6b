"""Non-square frame sizes (I2VGen-XL's native 1280 x 704, portrait 704 x 1280, 1024 x 576) without a GPU: the convolution tile plan
the dispatcher runs (av2v_conv3x3_plan, a host-only C-ABI call) for every 3x3 convolution of a UNet step and of the VAE, a
simulation of the epilogue's block-tile bookkeeping on those plans, and the pipeline's input check."""
import ctypes
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools import epilogue_schedule_model as esm  # noqa: E402
from tools import shape_census  # noqa: E402

# latent (height, width) of 512 x 512, 1280 x 704, 704 x 1280 and 1024 x 576 frames
LATENT_SIZES = [(64, 64), (88, 160), (160, 88), (72, 128)]


def _plan(g):
    from anyv2v_b200 import _lib
    a = _lib.GemmArgs()
    a.mode = _lib.A_CONV3X3
    for k in ("NF", "H", "W", "Cin", "N", "K", "M", "stride", "a_channels", "ldo", "n_slots", "up2_phase"):
        setattr(a, k, g[k])
    a.rowbias = 16 if g.get("rowbias") else None   # only tested for presence
    a.residual = 16 if g.get("residual") else None
    out = _lib.ConvPlan()
    rc = _lib.lib().av2v_conv3x3_plan(ctypes.byref(a), ctypes.byref(out))
    err = _lib.lib().av2v_last_error()
    return rc, (out.box_w, out.box_h, out.frames_per_tile, out.tiles_per_frame, out.m_tiles), (err.decode() if err else "")


def _conv(NF, H, W, Cin=320, N=320, stride=1, up2_phase=0, **kw):
    Ho, Wo = H // stride, W // stride
    g = dict(NF=NF, H=H, W=W, Cin=Cin, N=N, K=(4 if up2_phase else 9) * Cin, M=NF * Ho * Wo, stride=stride, a_channels=0, ldo=N,
             n_slots=1, up2_phase=up2_phase, residual=False, rowbias=False)
    g.update(kw)
    return g


@pytest.fixture(scope="module")
def census():
    """every distinct conv3x3 / up2-phase geometry of an inversion step (B = 1), an edit step (B = 3, conv + spatial + temporal
    injection) of the full-size UNet with 16 frames, and a VAE encode + decode of one frame, at each size"""
    geos = {}
    for h, w in LATENT_SIZES:
        calls = (shape_census.unet_conv_census(1, False, 16, h, w) + shape_census.unet_conv_census(3, True, 16, h, w)
                 + shape_census.vae_conv_census(1, 8 * h, 8 * w))
        for g in calls:
            geos[tuple(sorted(g.items()))] = g
    return list(geos.values())


def test_census_covers_the_native_resolution_levels(census):
    widths = {g["W"] // g["stride"] for g in census}
    assert {160, 80, 40, 20, 88, 44, 22, 11, 1280, 640, 320, 704, 352, 176}.issubset(widths)
    assert any(g["n_slots"] == 3 and g["W"] == 40 for g in census), "the 3-slot injection conv at the 40 x 22 level"
    assert any(g["up2_phase"] and g["W"] == 80 for g in census) and any(g["stride"] == 2 and g["W"] == 160 for g in census)


def test_every_census_conv_has_a_plan_that_covers_each_pixel_once(census):
    for g in census:
        rc, plan, err = _plan(g)
        assert rc == 0, (g, err)
        box_w, box_h, fpt, tpf, m_tiles = plan
        Ho, Wo = g["H"] // g["stride"], g["W"] // g["stride"]
        # TMA box limits: each box dimension <= 256 (the A box spans stride x the output block), at most 128 accumulator rows
        assert box_w * g["stride"] <= 256 and box_h * g["stride"] <= 256 and fpt <= 256, (g, plan)
        assert box_w * box_h * fpt <= 128, (g, plan)
        # simulate the tiles over two frames (the plan repeats per frame) or over all frames when a tile holds several
        nf = g["NF"] if fpt > 1 else min(g["NF"], 2)
        rc, plan_sim, err = _plan(dict(g, NF=nf, M=nf * Ho * Wo))
        assert rc == 0 and plan_sim[:4] == plan[:4], (g, plan, plan_sim)
        esm.check_block_tiles(plan_sim, nf, Ho, Wo, pair=True)


def test_native_resolution_plans_fill_their_tiles():
    # landscape 160 x 88 / 80 x 44 / 40 x 22 / 20 x 11 and portrait transposes: (box_w, box_h) and tile fill
    want = {(160, 88): (32, 4, 1.0), (80, 44): (16, 8, 0.917), (40, 22): (40, 3, 0.859), (20, 11): (20, 6, 0.859),
            (88, 160): (8, 16, 1.0), (44, 80): (16, 8, 0.917), (22, 40): (22, 5, 0.859), (11, 20): (11, 11, 0.859),
            (320, 176): (64, 2, 1.0), (704, 1280): (64, 2, 1.0), (352, 640): (32, 4, 1.0), (176, 320): (16, 8, 1.0),
            (88, 1280): (8, 16, 1.0)}
    for (W, H), (bw, bh, fill) in want.items():
        rc, plan, err = _plan(_conv(2, H, W))
        assert rc == 0, err
        assert plan[:3] == (bw, bh, 1), ((W, H), plan)
        assert abs(W * H / (plan[3] * 128) - fill) < 1e-3, ((W, H), plan, W * H / (plan[3] * 128))


def test_512_plans_are_unchanged():
    """512 x 512: the tile plans of the parent revision, hard-coded (box_w, box_h, frames_per_tile, m_tiles)."""
    cases = [  # UNet latent levels, 48 frames (edit step)
        (_conv(48, 64, 64), (64, 2, 1, 48 * 32)), (_conv(48, 32, 32, 640, 640), (32, 4, 1, 48 * 8)),
        (_conv(48, 16, 16, 1280, 1280), (16, 8, 1, 48 * 2)), (_conv(48, 8, 8, 1280, 1280), (8, 8, 2, 24)),
        (_conv(16, 64, 64, 64, 320, a_channels=8), (64, 2, 1, 16 * 32)),
        (_conv(16, 64, 64, stride=2), (32, 4, 1, 16 * 8)), (_conv(16, 16, 16, 1280, 1280, stride=2), (8, 8, 2, 8)),
        (_conv(16, 8, 8, 1280, 1280, up2_phase=1), (8, 8, 2, 8)), (_conv(16, 16, 16, 1280, 1280, up2_phase=4), (16, 8, 1, 32)),
        (_conv(16, 32, 32, 640, 640, up2_phase=2), (32, 4, 1, 16 * 8)),
        (_conv(48, 16, 16, 2560, 1280, n_slots=3, residual=True), (16, 8, 1, 96)),
        # VAE widths
        (_conv(1, 512, 512, 128, 128), (128, 1, 1, 2048)), (_conv(1, 256, 256, 256, 256), (128, 1, 1, 512)),
        (_conv(1, 128, 128, 512, 512), (128, 1, 1, 128)), (_conv(1, 64, 64, 512, 512), (64, 2, 1, 32)),
    ]
    for g, want in cases:
        rc, plan, err = _plan(g)
        assert rc == 0, (g, err)
        assert (plan[0], plan[1], plan[2], plan[4]) == want, (g, plan, want)


def test_width_160_is_accepted():
    """conv_in / the finest resnet convs at 1280 x 704: width 160 (before block tiles only widths <= 128 or multiples of 128 ran;
    av2v_gemm_f16 returned AV2V_ENOSUP for this geometry)"""
    for g in (_conv(16, 88, 160, 64, 320, a_channels=8), _conv(16, 88, 160, rowbias=True), _conv(48, 88, 160, residual=True),
              _conv(16, 176, 320, stride=2), _conv(16, 80, 80, up2_phase=3)):
        rc, plan, err = _plan(g)
        assert rc == 0, (g, err)


def test_plan_rejects_what_the_kernel_cannot_run():
    from anyv2v_b200 import _lib
    assert _plan(_conv(2, 88, 160, Cin=96))[0] == _lib.AV2V_ENOSUP          # Cin not a multiple of 64
    assert _plan(_conv(2, 87, 160, stride=2))[0] == _lib.AV2V_ENOSUP        # odd height with stride 2
    assert _plan(dict(_conv(2, 88, 160), M=5))[0] == _lib.AV2V_EINVAL       # M != NF * H * W
    assert _plan(_conv(2, 22, 40, up2_phase=1, ldo=640))[0] == _lib.AV2V_ENOSUP  # up2 needs a contiguous output


def test_conv_plan_struct_matches_the_c_header_layout(tmp_path):
    from anyv2v_b200 import _lib
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "anyv2v_b200.h"', 'int main(void) {',
             '  printf("size %zu\\n", sizeof(av2v_conv_plan));']
    for fname, _ in _lib.ConvPlan._fields_:
        lines.append(f'  printf("{fname} %zu\\n", offsetof(av2v_conv_plan, {fname}));')
    lines += ['  return 0;', '}']
    src = tmp_path / "plan_probe.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "plan_probe"
    subprocess.run(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    out = dict(l.split() for l in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    assert int(out["size"]) == ctypes.sizeof(_lib.ConvPlan)
    for fname, _ in _lib.ConvPlan._fields_:
        assert int(out[fname]) == getattr(_lib.ConvPlan, fname).offset, fname


def test_epilogue_model_block_tiles():
    """the epilogue's tile origin + per-row pixel on block tiles, including edge blocks, whole-frame tiles and the phantom tile of
    a CTA pair when m_tiles is odd"""
    for W, H, NF in ((160, 88, 3), (88, 160, 1), (80, 44, 3), (40, 22, 3), (22, 40, 1), (20, 11, 5), (11, 20, 3), (24, 20, 2),
                     (320, 176, 1), (12, 4, 7), (64, 64, 2)):
        rc, plan, err = _plan(_conv(NF, H, W))
        assert rc == 0, err
        esm.check_block_tiles(plan, NF, H, W, pair=True)
    # a plan with too few row blocks per frame leaves the bottom rows unwritten: the check must see it
    with pytest.raises(AssertionError):
        esm.check_block_tiles((40, 3, 1, 7, 21), 3, 22, 40)  # 7 row blocks of 3 rows leave row 21 uncovered
    # the lean epilogue's chunk bookkeeping is unchanged by the tile shape: a block plan's m_tiles as the M units
    esm.check(0, 148, 330, 2, 320, 160, False)
    esm.check(5, 74, 165, 2, 320, 160, False)


def test_check_inputs_rejects_latents_not_divisible_by_the_unet_depth():
    from types import SimpleNamespace
    from anyv2v_b200.pipeline import I2VGenXLPipeline
    from anyv2v_b200.unet_i2vgen_xl import I2VGEN_XL_CONFIG
    pipe = I2VGenXLPipeline(SimpleNamespace(config=dict(I2VGEN_XL_CONFIG)))
    z = lambda h, w: torch.zeros(1, 4, 2, h, w)
    e = torch.zeros(1, 77, 1024)
    with pytest.raises(ValueError, match="multiples of 64 px"):
        pipe.check_inputs(e, z(90, 160), e, z(90, 160))
    pipe.check_inputs(e, z(88, 160), e, z(88, 160))
    pipe.check_inputs(e, z(160, 88), e, z(160, 88))
    tiny = I2VGenXLPipeline(SimpleNamespace(config=dict(I2VGEN_XL_CONFIG, block_out_channels=(64, 128))))
    tiny.check_inputs(e, z(6, 10), e, z(6, 10))  # two levels: multiples of 2 are enough

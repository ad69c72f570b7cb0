"""GPU parity against the REFERENCE ITSELF (the unmodified timg translation units), one hop instead of two: the
CUDA path is compared with what ImageScaler::Scale, Framebuffer::AlphaComposeBackground and UnicodeBlockCanvas::Send
produced at the geometries of BASELINE.json's configs, including multi-frame batches (>= 64 frames for C3 / C4 /
C5) and C3's scaling + delta emission together.  Those outputs are too large for the repository, so
tests/golden/reference_configs.npz keeps their sha256 digests (written by tests/golden/make_golden.py).
"""
import os

import numpy as np
import pytest

import cases
import oracle
import timg_b200
from timg_b200 import synth

pytestmark = pytest.mark.gpu

BG = oracle.rgba_u32(0, 0, 0)


@pytest.fixture(scope="module")
def golden():
    return np.load(os.path.join(os.path.dirname(__file__), "golden", "reference_configs.npz"))


def _batch(n, iw, ih, ow, oh, **kw):
    d = dict(n_frames=n, src_w=iw, src_h=ih, src_fmt=0, out_w=ow, out_h=oh, has_bg=1, bg=BG, pattern=0, pattern_w=0,
             pattern_h=0, flags=0, x_indent_cells=0, animation=0)
    d.update(kw)
    return timg_b200.Batch(**d)


@pytest.mark.parametrize("iw,ih,fit,kind", cases.CONFIG_GEOMETRIES)
def test_scaler_and_compose_equal_the_reference_at_config_geometries(ctx, golden, iw, ih, fit, kind):
    _, ow, oh = timg_b200.calc_fit(iw, ih, *fit)
    got = ctx.scale(cases.config_image(iw, ih, kind), ow, oh)
    assert cases.digest(got) == golden[f"scale_{iw}x{ih}_{ow}x{oh}"]
    assert cases.digest(ctx.compose_bg(got, BG)) == golden[f"compose_{iw}x{ih}_{ow}x{oh}"]


def test_c1_half_blocks_batch_equals_reference_canvas(ctx, golden):
    n, iw, ih = cases.CONFIG_BATCH, 640, 480
    _, ow, oh = timg_b200.calc_fit(iw, ih, 80, 50, 1, 2)
    outs = ctx.blocks_batch(cases.c1_frames(), _batch(n, iw, ih, ow, oh))
    for f in range(n):
        assert cases.digest(outs[f]) == golden["c1_half"][f], f


def test_c3_quarter_animation_scale_plus_delta_equals_reference_canvas(ctx, golden):
    """C3: 1080p -> 320x90 -> -p quarter, 64 frames, frame 0 full and the rest emitted as differences, scaling and
    delta emission in ONE batch call, against the reference's scaler + compose + ONE stateful UnicodeBlockCanvas."""
    n, iw, ih = cases.CONFIG_BATCH, 1920, 1080
    _, ow, oh = timg_b200.calc_fit(iw, ih, 320, 100, 2, 2, 2.0)
    assert (ow, oh) == (320, 90)
    outs = ctx.blocks_batch(cases.c3_frames(), _batch(n, iw, ih, ow, oh, flags=timg_b200.QUARTER, animation=1))
    for f in range(n):
        prefix = b"" if f == 0 else b"\033[%dA" % (oh // 2)      # the adapter adds the cursor-up, the ABI returns image bytes
        assert cases.digest(prefix + outs[f]) == golden["c3_quarter_delta"][f], f
    assert sum(len(o) for o in outs[1:]) < len(outs[0]) * (n - 1) // 4      # deltas really are deltas


def test_c4_grid_sixel_batch_of_64_equals_staged_reference_scaler(ctx, golden):
    """C4: 64 distinct 4K frames -> 337x190 (+pad 192) sixel in one batch == reference scaler + compose per frame,
    then the single-frame encoder (whose own parity is covered in test_sixel_gpu.py).  The staged frames are
    rebuilt with the CPU restatements and must hash to the reference's own."""
    n, iw, ih = cases.CONFIG_BATCH, 3840, 2160
    _, ow, oh = timg_b200.calc_fit(iw, ih, 337, 225, 9, 18)
    frames = cases.c4_frames()
    outs = ctx.sixel_batch(frames, _batch(n, iw, ih, ow, oh))
    hp = (oh + 5) // 6 * 6
    for f in range(n):
        fb = np.zeros((hp, ow, 4), np.uint8)
        fb[:oh] = oracle.compose_bg(oracle.stb_resize(frames[f], ow, oh), BG)
        fb = oracle.compose_bg(fb, BG, start_row=oh)                        # SixelCanvas::Send's pad strip
        assert cases.digest(fb) == golden["c4_staged"][f], f
        assert outs[f] == ctx.sixel_encode(fb), f


def test_c5_unscaled_720p_sixel_batch_of_64(ctx):
    n, w, h = 64, 1280, 720
    frames = cases.variants(np.stack([synth.frame_np(200 + i, w, h, "photo") for i in range(8)]), n)
    outs = ctx.sixel_batch(frames, _batch(n, w, h, w, h))
    for f in range(0, n, 7):                                               # every 7th frame against the CPU restatement (0.1 s each)
        img, used = oracle.sixel_decode(outs[f])
        want, _ = oracle.sixel_decode(oracle.sixel_encode(frames[f], mode=1))
        assert (img == want).all(), f
    assert len({o for o in outs}) > n // 2                                 # the frames really are distinct

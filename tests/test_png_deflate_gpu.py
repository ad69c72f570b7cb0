"""The compressed PNG behind the kitty / iTerm2 canvases (timg_b200/csrc/deflate.cu): timg's --compress level.

Reference: png::Encode, src/timg-png.cc:90-152, deflating with libdeflate at DisplayOptions::compress_pixel_level
(1 by default).  libdeflate is third party, so parity is the same as for the stored path: the stream parses with
Python's zlib, every CRC and the Adler-32 verify, each row is Sub-filtered and the pixels are the source's.  On top:
the zlib header is well formed, sizes stay within the bound and near zlib -1, a batch slice equals the one-frame
call, and the batch keeps the output capacity contract of the other *_dev calls.
"""
import base64
import ctypes as C
import zlib

import numpy as np
import pytest

import timg_b200
from timg_b200 import synth
from test_png_gpu import png_decode

SEG = 16384                     # filtered bytes per deflate segment (deflate.cu DF_SEG)


def flat_graphic(w, h, seed=5):
    """Palette blocks with dark one-pixel 'text' lines: the content LZ77 with history carries."""
    rng = np.random.default_rng(seed)
    pal = rng.integers(0, 256, (12, 4), dtype=np.uint8)
    pal[:, 3] = 255
    bw, bh = 90, 60
    idx = rng.integers(0, len(pal), ((h + bh - 1) // bh, (w + bw - 1) // bw))
    fb = pal[np.repeat(np.repeat(idx, bh, 0), bw, 1)[:h, :w]].copy()
    for y in range(8, h, 17):
        x0 = int(rng.integers(0, max(1, w // 2)))
        fb[y, x0:x0 + int(rng.integers(20, max(21, w // 3))), :3] = 20
    return fb


def filtered(fb, rgb24):
    """The Sub-filtered scanline stream png.cu defines (filter byte 1 per row)."""
    px = fb[..., :3] if rgb24 else fb
    h, w, bpp = px.shape
    d = px.astype(np.int16)
    d[:, 1:] -= px[:, :-1]
    rows = np.concatenate([np.ones((h, 1), np.uint8), (d & 255).astype(np.uint8).reshape(h, w * bpp)], axis=1)
    return rows.tobytes()


def check_zlib(data):
    """zlib header fields and a stream that ends exactly where IDAT ends."""
    n = int.from_bytes(data[33:37], "big")
    z = data[41:41 + n]
    cmf, flg = z[0], z[1]
    assert cmf & 15 == 8 and cmf >> 4 == 7 and not flg & 0x20 and (cmf * 256 + flg) % 31 == 0
    d = zlib.decompressobj(wbits=15)
    d.decompress(z)
    assert d.eof and d.unused_data == b""


def encode_ok(ctx, fb, rgb24, level):
    h, w = fb.shape[:2]
    data, b64 = ctx.png_encode(fb, rgb24, level=level)
    assert len(data) <= timg_b200.lib().b200timg_png_bound(w, h, int(rgb24), level)
    px, ctype = png_decode(data)
    assert ctype == (2 if rgb24 else 6)
    assert (px == (fb[..., :3] if rgb24 else fb)).all()
    check_zlib(data)
    assert b64 == base64.b64encode(data)
    return data


SHAPES = [(67, 50, "alpha"), (1, 1, "noise"), (320, 90, "photo"), (333, 201, "noisea"), (2700, 25, "photo"),
          (16390, 4, "noise")]


@pytest.mark.gpu
@pytest.mark.parametrize("level", [1, 9])
@pytest.mark.parametrize("w,h,kind", SHAPES)
def test_deflate_decodes_to_the_source_pixels(ctx, w, h, kind, level):
    fb = synth.frame_np(3 + w, w, h, kind)
    for rgb24 in (False, True):
        encode_ok(ctx, fb, rgb24, level)


@pytest.mark.gpu
@pytest.mark.parametrize("level", [1, 9])
def test_deflate_special_lengths(ctx, level):
    const = np.full((70, 300, 4), 77, np.uint8)                      # maximal overlapping matches
    small = synth.frame_np(9, 40, 30, "photo")                        # shorter than one segment
    # filtered length an exact multiple of the segment size: RGBA rows of 1 + 4 * 4095 = 16381 bytes do not divide,
    # RGB rows of 1 + 3 * 5461 = 16384 bytes do
    multiple = synth.frame_np(11, 5461, 3, "photo")
    assert len(filtered(multiple, True)) == 3 * SEG
    for fb, modes in ((const, (False, True)), (small, (False, True)), (multiple, (True,))):
        for rgb24 in modes:
            data = encode_ok(ctx, fb, rgb24, level)
            if fb is const:
                assert len(data) < 200 + len(filtered(fb, rgb24)) // 100


@pytest.mark.gpu
@pytest.mark.parametrize("level", [1, 9])
def test_deflate_flat_graphic_c2_size_decodes(ctx, level):
    fb = flat_graphic(2700, 1519)
    for rgb24 in (False, True):
        encode_ok(ctx, fb, rgb24, level)


@pytest.mark.gpu
def test_deflate_level0_is_the_stored_path(ctx):
    L = timg_b200.lib()
    for w, h, kind in SHAPES[:4]:
        fb = synth.frame_np(3 + w, w, h, kind)
        for rgb24 in (0, 1):
            want = ctx.png_encode(fb, bool(rgb24))
            n = L.b200timg_png_bound(w, h, rgb24, 0)
            out = np.zeros(n, np.uint8)
            b64 = C.create_string_buffer(L.b200timg_base64_size(n))
            got = C.c_size_t()
            rc = L.b200timg_png_encode_level(ctx.h, fb.ctypes.data_as(timg_b200.u8p), w, h, rgb24, 0,
                                             out.ctypes.data_as(timg_b200.u8p), n, C.byref(got), b64, len(b64))
            assert rc == timg_b200.OK and got.value == n
            assert out.tobytes() == want[0] and b64.raw == want[1]
            assert ctx.png_encode(fb, bool(rgb24), level=0) == want


@pytest.mark.gpu
def test_deflate_rejects_levels_outside_0_to_9(ctx):
    fb = synth.frame_np(1, 8, 8, "photo")
    for level in (-1, 10):
        with pytest.raises(timg_b200.B200Error) as e:
            ctx.png_encode(fb, level=level)
        assert e.value.code == timg_b200.EINVAL


@pytest.mark.gpu
def test_deflate_size_against_zlib1(ctx):
    w, h = 2700, 1519
    photo = synth.frame_np(17, w, h, "photo")
    flat = flat_graphic(w, h)
    for fb, factor in ((photo, 1.02), (flat, 1.5)):
        data = encode_ok(ctx, fb, False, 1)
        z1 = len(zlib.compress(filtered(fb, False), 1))
        assert len(data) - 57 <= factor * z1, (len(data), z1)
    noise = synth.frame_np(4, 640, 360, "noise")
    for rgb24 in (False, True):
        data = encode_ok(ctx, noise, rgb24, 1)
        assert len(data) <= timg_b200.lib().b200timg_png_size(640, 360, int(rgb24))


def _batch(ctx, frames, rgb24, level, png_cap=None, b64_cap=None, guard=64):
    import torch
    n, h, w = frames.shape[:3]
    L = timg_b200.lib()
    bound = L.b200timg_png_bound(w, h, int(rgb24), level)
    png_cap = n * bound if png_cap is None else png_cap
    b64_cap = n * L.b200timg_base64_size(bound) if b64_cap is None else b64_cap
    d_frames = torch.from_numpy(frames).cuda()
    d_png = torch.full((png_cap + guard,), 0xA5, dtype=torch.uint8, device="cuda")
    d_b64 = torch.full((b64_cap + guard,), 0xA5, dtype=torch.uint8, device="cuda")
    d_off = torch.zeros(n + 1, dtype=torch.int64, device="cuda")
    d_boff = torch.zeros(n + 1, dtype=torch.int64, device="cuda")
    rc = L.b200timg_png_batch_level_dev(ctx.h, d_frames.data_ptr(), w, h, n, int(rgb24), level, d_png.data_ptr(), png_cap,
                                        d_off.data_ptr(), d_b64.data_ptr(), b64_cap, d_boff.data_ptr())
    assert rc == timg_b200.OK, L.b200timg_last_error(ctx.h)
    torch.cuda.synchronize()
    return d_png.cpu().numpy(), d_b64.cpu().numpy(), d_off.cpu().numpy(), d_boff.cpu().numpy()


def _mixed(n, w, h):
    kinds = ["photo", "noise", "alpha", "noisea"]
    frames = [synth.frame_np(30 + i, w, h, kinds[i % 4]) for i in range(n)]
    frames[2] = flat_graphic(w, h, seed=2)
    frames[-1] = np.full((h, w, 4), 200, np.uint8)
    return np.stack(frames)


@pytest.mark.gpu
@pytest.mark.parametrize("rgb24", [False, True])
def test_deflate_batch_slices_equal_single_frames(ctx, rgb24):
    n, w, h = 7, 301, 123
    frames = _mixed(n, w, h)
    png, b64, off, boff = _batch(ctx, frames, rgb24, 1)
    for f in range(n):
        data, text = ctx.png_encode(frames[f], rgb24, level=1)
        assert png[off[f]:off[f + 1]].tobytes() == data
        assert b64[boff[f]:boff[f + 1]].tobytes() == text == base64.b64encode(data)
    assert (png[off[n]:] == 0xA5).all() and (b64[boff[n]:] == 0xA5).all()


@pytest.mark.gpu
@pytest.mark.parametrize("level", [0, 1])
def test_deflate_batch_too_small_buffer_keeps_the_capacity_contract(ctx, level):
    n, w, h = 5, 200, 90
    frames = _mixed(n, w, h)
    _, _, off, boff = _batch(ctx, frames, False, level)
    cap = int(off[3]) - 1                                           # frames 0, 1 fit; 2 ends one byte beyond
    png, b64, off2, boff2 = _batch(ctx, frames, False, level, png_cap=cap)
    assert (off2 == off).all() and (boff2 == boff).all()           # offsets complete and exact
    for f in range(2):
        data, text = ctx.png_encode(frames[f], False, level=level)
        assert png[off[f]:off[f + 1]].tobytes() == data
        assert b64[boff[f]:boff[f + 1]].tobytes() == text
    assert (png[off[2]:] == 0xA5).all()                            # later frames and the guard bytes untouched
    assert (b64[boff[2]:] == 0xA5).all()


@pytest.mark.gpu
def test_deflate_single_frame_too_small_reports_the_need(ctx):
    L = timg_b200.lib()
    fb = flat_graphic(300, 200)
    data, _ = ctx.png_encode(fb, level=1)
    out = np.full(len(data) + 16, 0xA5, np.uint8)
    got = C.c_size_t()
    rc = L.b200timg_png_encode_level(ctx.h, fb.ctypes.data_as(timg_b200.u8p), 300, 200, 0, 1, out.ctypes.data_as(timg_b200.u8p),
                                     len(data) - 1, C.byref(got), None, 0)
    assert rc == timg_b200.ENOSPC and got.value == len(data) and (out == 0xA5).all()


def test_png_bound_is_host_only_and_tight():
    L = timg_b200.lib()
    for w, h in ((1, 1), (67, 50), (333, 201), (2700, 1519), (16390, 4), (5461, 3), (1920, 1080)):
        for rgb24 in (0, 1):
            size = L.b200timg_png_size(w, h, rgb24)
            assert L.b200timg_png_bound(w, h, rgb24, 0) == size
            for level in range(1, 10):
                bound = L.b200timg_png_bound(w, h, rgb24, level)
                assert size <= bound <= size * 1.002 + 64

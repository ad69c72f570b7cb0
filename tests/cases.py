"""Deterministic input cases for the block-mode / compose parity tests (SURVEY.md App. C).

Every case is (name, dict) where the dict has: frames (list of HxWx4 uint8 arrays sent
one after another to ONE canvas), quarter/upper/color8 flags, x indent in pixels and the
dy passed for frames after the first (-height = animation / delta mode, 0 = fresh frame).
"""
import hashlib

import numpy as np

from timg_b200 import synth


def _solid(w, h, rgba):
    a = np.empty((h, w, 4), np.uint8)
    a[:] = np.array(rgba, np.uint8)
    return a


def _digits_frame(w, h):
    vals = np.array([0, 9, 10, 99, 100, 255, 1, 254, 47, 48, 114, 115, 154, 155, 194, 195, 234, 235], np.uint8)
    rng = np.random.default_rng(7)
    a = vals[rng.integers(0, len(vals), (h, w, 4))]
    a[..., 3] = 255
    return a


def _quarter_patterns():
    """2x2 cells exercising every partition, near ties and the d<1 early break."""
    A, B = (200, 30, 40, 255), (20, 220, 90, 255)
    C, D = (201, 30, 40, 255), (200, 31, 40, 255)
    cells = []
    for mask in range(16):          # which of tl,tr,bl,br take colour B
        cells.append([B if mask & (1 << k) else A for k in range(4)])
    cells.append([A, C, A, C]); cells.append([A, A, C, C]); cells.append([A, C, C, A])
    cells.append([A, D, C, A]); cells.append([A, A, A, C]); cells.append([C, A, A, A])
    cells.append([(0, 0, 0, 255), (1, 1, 1, 255), (0, 0, 0, 255), (1, 1, 1, 255)])
    cells.append([(255, 255, 255, 255), (254, 255, 255, 255), (255, 254, 255, 255), (255, 255, 254, 255)])
    T, U = (10, 20, 30, 0x20), (40, 50, 60, 0x5f)      # transparent (a < 0x60)
    S = (90, 80, 70, 0x60)                              # just opaque enough
    cells += [[T, U, A, B], [A, B, T, U], [T, U, U, T], [T, A, U, B], [A, T, B, U], [S, T, T, S],
              [(100, 100, 100, 0x5f), (100, 100, 100, 0x61), A, A],
              [(100, 100, 100, 0xbf), (50, 50, 50, 0x00), (30, 30, 30, 0x00), (20, 20, 20, 0x00)]]
    n = len(cells)
    per_row = 8
    rows = (n + per_row - 1) // per_row
    a = np.zeros((rows * 2, per_row * 2, 4), np.uint8)
    a[..., 3] = 255
    for i, (tl, tr, bl, br) in enumerate(cells):
        r, c = divmod(i, per_row)
        a[2 * r, 2 * c] = tl; a[2 * r, 2 * c + 1] = tr
        a[2 * r + 1, 2 * c] = bl; a[2 * r + 1, 2 * c + 1] = br
    return a


def _runs_frame(w, h):
    """same-fg runs with intervening space glyphs, same-bg runs, transparent cells."""
    a = _solid(w, h, (10, 20, 30, 255))
    a[1::2, 2:6] = (200, 100, 50, 255)       # fg cells (bottom differs)
    a[1::2, 8:10] = (200, 100, 50, 255)      # same fg again after spaces
    a[0::2, 12:14] = (1, 2, 3, 255)          # bg changes, fg stays
    a[:, 16:18] = (0, 0, 0, 0)               # fully transparent cells -> "49;"
    a[0::2, 20:22] = (5, 5, 5, 0x10)         # top transparent only
    return a


def block_cases():
    cases = []
    for q in (0, 1):
        for up in (0, 1):
            for c8 in (0, 1):
                tag = f"q{q}u{up}c{c8}"
                w, h = (66, 50) if q else (67, 50)
                cases.append((f"noisea_{tag}", dict(frames=[synth.frame_np(11, w, h, "noisea")], quarter=q,
                                                    upper=up, color8=c8, x=0, dy=0)))
                cases.append((f"photo_odd_{tag}", dict(frames=[synth.frame_np(12, w, 37, "photo")], quarter=q,
                                                       upper=up, color8=c8, x=6, dy=0)))
                cases.append((f"digits_{tag}", dict(frames=[_digits_frame(40, 14)], quarter=q, upper=up,
                                                    color8=c8, x=0, dy=0)))
                cases.append((f"runs_{tag}", dict(frames=[_runs_frame(24, 9)], quarter=q, upper=up, color8=c8,
                                                  x=4, dy=0)))
                cases.append((f"qpat_{tag}", dict(frames=[_quarter_patterns()], quarter=q, upper=up, color8=c8,
                                                  x=0, dy=0)))
    # delta sequences (SURVEY App. D and friends)
    for q in (0, 1):
        for up in (0, 1):
            tag = f"q{q}u{up}"
            base = _solid(4, 16, (10, 20, 30, 255))
            f2 = base.copy(); f2[13, 2] = (200, 100, 50, 255)
            f3 = f2.copy()
            f4 = f3.copy(); f4[2, 0] = (1, 2, 3, 255); f4[3, 3] = (1, 2, 3, 255)
            cases.append((f"delta_appD_{tag}", dict(frames=[base, f2, f3, f4], quarter=q, upper=up, color8=0,
                                                    x=0, dy=-16)))
            # empty-row runs of 1..6 between changed rows, trailing empties, odd height
            h = 61
            seq = [synth.frame_np(21, 32, h, "photo")]
            cur = seq[0].copy()
            for step, rows in enumerate([(0,), (2, 6), (6, 16), (16, 28), (28, 42), (1, 59), ()]):
                cur = cur.copy()
                for r in rows:
                    cur[r, (3 * step) % 30:(3 * step) % 30 + 2] = (step * 30 % 256, 255 - step * 20, 7, 255)
                seq.append(cur)
            cases.append((f"delta_rows_{tag}", dict(frames=seq, quarter=q, upper=up, color8=0, x=2 * (1 + q),
                                                    dy=-h)))
            # moving sprite animation
            seq = []
            for k in range(6):
                fr = synth.frame_np(31, 64, 40, "photo")
                fr[5 + 2 * k:13 + 2 * k, 8 + 5 * k:16 + 5 * k] = synth.frame_np(40 + k, 8, 8, "noise")
                seq.append(fr)
            cases.append((f"delta_sprite_{tag}", dict(frames=seq, quarter=q, upper=up, color8=1 - q, x=0,
                                                      dy=-40)))
    # a fresh (dy=0) second frame must be emitted in full even if identical
    fr = synth.frame_np(51, 20, 10, "photo")
    cases.append(("fresh_second_frame", dict(frames=[fr, fr.copy()], quarter=0, upper=0, color8=0, x=0, dy=0)))
    # C1-shaped frame: 640x480 -> 67x50 half (config 0 of BASELINE.json), as random + alpha variants
    cases.append(("c1_random", dict(frames=[synth.frame_np(1234, 67, 50, "noisea")], quarter=0, upper=0,
                                    color8=0, x=0, dy=0)))
    cases.append(("c1_photo", dict(frames=[synth.frame_np(1234, 67, 50, "photo")], quarter=0, upper=0,
                                   color8=0, x=0, dy=0)))
    return cases


def compose_cases():
    """(name, fb, kwargs) for AlphaComposeBackground."""
    from timg_b200 import rgba_u32
    bg, pat = rgba_u32(30, 60, 200), rgba_u32(200, 180, 20)
    out = []
    fa = synth.frame_np(61, 53, 31, "noisea")
    edge = fa.copy()
    edge[0, :8, 3] = [0, 1, 254, 255, 0x5f, 0x60, 128, 127]
    out.append(("noisea_plain", fa, dict(bg=bg)))
    out.append(("noisea_checker", fa, dict(bg=bg, pattern=pat, pw=3, ph=2)))
    out.append(("noisea_checker_half", fa, dict(bg=bg, pattern=pat, pw=1, ph=1)))
    out.append(("edge_alpha", edge, dict(bg=bg, pattern=pat, pw=2, ph=2)))
    out.append(("start_row", fa, dict(bg=bg, pattern=pat, pw=4, ph=3, start_row=17)))
    out.append(("pattern_equals_bg", fa, dict(bg=bg, pattern=bg, pw=4, ph=3)))
    out.append(("pattern_transparent", fa, dict(bg=bg, pattern=rgba_u32(1, 2, 3, 0), pw=4, ph=3)))
    out.append(("bg_transparent", fa, dict(bg=rgba_u32(9, 9, 9, 0), pattern=pat, pw=4, ph=3)))
    out.append(("no_bg", fa, dict(bg=bg, has_bg=False)))
    out.append(("opaque", synth.frame_np(62, 40, 20, "photo"), dict(bg=bg, pattern=pat, pw=2, ph=2)))
    out.append(("alpha_checker_img", synth.frame_np(63, 128, 96, "alpha"), dict(bg=rgba_u32(0, 0, 0), pattern=pat,
                                                                                pw=8, ph=4)))
    out.append(("white_bg", fa, dict(bg=rgba_u32(255, 255, 255))))
    out.append(("odd_size", synth.frame_np(64, 7, 3, "noisea"), dict(bg=bg, pattern=pat, pw=2, ph=1)))
    return out


def run_block_case(make_canvas, case):
    """Send the case's frames through a canvas factory (quarter, upper, color8) -> object with
    .send(fb, x, dy).  Returns list of bytes."""
    cv = make_canvas(case["quarter"], case["upper"], case["color8"])
    outs = []
    for i, fr in enumerate(case["frames"]):
        outs.append(cv.send(fr, case["x"], 0 if i == 0 else case["dy"]))
    return outs


def digest(data):
    """sha256 of an array's or a byte string's bytes: how outputs too large to store are kept as golden data."""
    if isinstance(data, np.ndarray):
        data = np.ascontiguousarray(data).tobytes()
    return hashlib.sha256(data).hexdigest()


def random_block_case(seed):
    """A small random frame and three sparse deltas, random canvas flags."""
    rng = np.random.default_rng(100 + seed)
    q, up, c8 = int(rng.integers(0, 2)), int(rng.integers(0, 2)), int(rng.integers(0, 2))
    w = int(rng.integers(1, 60)) * (2 if q else 1)
    h = int(rng.integers(1, 50))
    kind = ["noisea", "photo", "alpha", "noise"][seed % 4]
    frames = [synth.frame_np(1000 + seed, w, h, kind)]
    for k in range(3):                      # sparse deltas
        f = frames[-1].copy()
        ys, xs = rng.integers(0, h, 5), rng.integers(0, w, 5)
        f[ys, xs] = rng.integers(0, 256, (5, 4), dtype=np.uint8)
        frames.append(f)
    return dict(frames=frames, quarter=q, upper=up, color8=c8, x=int(rng.integers(0, 9)), dy=-h)


def random_compose_cases():
    """(fb, kwargs) for AlphaComposeBackground with random sizes, colours, patterns and start rows."""
    rng = np.random.default_rng(9)
    out = []
    for i in range(10):
        w, h = int(rng.integers(1, 80)), int(rng.integers(1, 60))
        fb = synth.frame_np(300 + i, w, h, "noisea")
        kw = dict(bg=int(rng.integers(0, 2 ** 24)) | 0xff000000, pattern=int(rng.integers(0, 2 ** 32)),
                  pw=int(rng.integers(0, 5)), ph=int(rng.integers(0, 5)), start_row=int(rng.integers(0, h)))
        out.append((fb, kw))
    return out


def as256_values():
    """RGBA words for the 256-colour mapping: random ones plus every threshold of the colour cube and grey ramp."""
    from timg_b200 import rgba_u32
    rng = np.random.default_rng(3)
    vals = list(rng.integers(0, 2 ** 32, 20000, dtype=np.uint64))
    for r in (0, 46, 47, 48, 114, 115, 154, 155, 194, 195, 234, 235, 255):
        for g in (0, 47, 115, 255):
            vals.append(rgba_u32(r, g, r))
            vals.append(rgba_u32(r, r, r))
    return [int(v) for v in vals]


def random_scale_cases():
    """(img, ow, oh, fmt) for ImageScaler::Scale: random sizes, arbitrary / integer / one-axis up- and downscales."""
    rng = np.random.default_rng(2)
    out = []
    for it in range(120):
        iw, ih = int(rng.integers(1, 300)), int(rng.integers(1, 200))
        mode = it % 5
        if mode == 0:
            ow, oh = int(rng.integers(1, 300)), int(rng.integers(1, 200))
        elif mode == 1:
            ow, oh = max(1, iw // int(rng.integers(1, 9))), max(1, ih // int(rng.integers(1, 9)))
        elif mode == 2:
            ow, oh = iw * int(rng.integers(1, 4)), ih * int(rng.integers(1, 4))
        elif mode == 3:
            ow, oh = iw, int(rng.integers(1, 200))
        else:
            ow, oh = int(rng.integers(1, 300)), ih
        img = synth.frame_np(it, iw, ih, ["noisea", "photo", "alpha", "noise"][it % 4])
        if it % 7 == 0:
            img[: ih // 2, :, 3] = 0
        out.append((img, ow, oh, it % 2))
    return out


# ---- BASELINE.json's config geometries, as the GPU tests against the reference's own outputs run them
CONFIG_GEOMETRIES = [(640, 480, (80, 50, 1, 2, 1.0), "alpha"),            # C1
                     (3840, 2160, (2700, 1800, 9, 18, 1.0), "photo"),       # C2
                     (1920, 1080, (320, 100, 2, 2, 2.0), "photo"),          # C3
                     (3840, 2160, (337, 225, 9, 18, 1.0), "alpha"),         # C4
                     (1280, 720, (2700, 1800, 9, 18, 1.0), "photo")]       # C5
CONFIG_BATCH = 64


def config_image(iw, ih, kind):
    return synth.frame_np(11 + iw, iw, ih, kind)


def variants(base, n):
    """n distinct frames from a few generated ones (cheap: a per-frame byte rotation of the colour channels)."""
    out = np.empty((n,) + base.shape[1:], np.uint8)
    for f in range(n):
        fr = base[f % len(base)].copy()
        fr[..., :3] = fr[..., :3] + np.uint8((37 * (f // len(base))) & 255)
        out[f] = fr
    return out


def c1_frames():
    """C1: 64 distinct 640x480 frames (alpha and noise)."""
    return variants(np.stack([synth.frame_np(500 + i, 640, 480, "alpha" if i % 2 else "noise") for i in range(8)]),
                    CONFIG_BATCH)


def c3_frames():
    """C3: 64 1080p frames, a photo base with a 64x64 noise sprite moving across it."""
    iw, ih = 1920, 1080
    base = synth.frame_np(77, iw, ih, "photo")
    frames = np.repeat(base[None], CONFIG_BATCH, 0)
    for k in range(CONFIG_BATCH):
        x, y = (37 + 8 * k) % (iw - 64), (91 + 5 * k) % (ih - 64)
        frames[k, y:y + 64, x:x + 64] = synth.frame_np(1077 + k, 64, 64, "noise")
    return frames


def c4_frames():
    """C4: 64 distinct 4K photo frames."""
    return variants(np.stack([synth.frame_np(900 + i, 3840, 2160, "photo") for i in range(4)]), CONFIG_BATCH)


def scale_cases():
    """(name, img, ow, oh, fmt) for ImageScaler::Scale parity (SURVEY App. C 'scaler' row)."""
    out = []
    geos = [("c1_640x480_to_67x50", 640, 480, 67, 50), ("identity", 61, 47, 61, 47), ("up2", 40, 30, 80, 60),
            ("up3", 21, 17, 63, 51), ("up_nonint", 37, 23, 80, 51), ("down_nonint", 200, 150, 141, 106),
            ("down_h_only", 200, 60, 77, 60), ("down_v_only", 120, 200, 120, 33), ("to_1x1", 17, 9, 1, 1),
            ("to_1xN", 50, 40, 1, 13), ("c3_ratio_1080p", 384, 216, 64, 18), ("c2_ratio_45_64", 256, 144, 180, 101),
            ("extreme_down", 1000, 30, 20, 3), ("mixed_up_down", 30, 300, 90, 40), ("tall_scatter", 12, 400, 12, 9)]
    for name, iw, ih, ow, oh in geos:
        for kind in ("noisea", "photo"):
            img = synth.frame_np(iw * 31 + ih, iw, ih, kind)
            if kind == "noisea":
                img[: ih // 3, :, 3] = 0                   # alpha=0 region keeps RGB (fancy alpha)
            out.append((f"{name}_{kind}", img, ow, oh, 0))
    img = synth.frame_np(99, 90, 70, "alpha")
    out.append(("bgra_down", img, 45, 31, 1))
    out.append(("bgra_identity", img, 90, 70, 1))
    return out

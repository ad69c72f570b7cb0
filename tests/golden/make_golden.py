"""Regenerates tests/golden/*.npz from the reference itself (oracle/_ref/libtimg_ref.so, i.e. the
UNMODIFIED timg translation units compiled by oracle/Makefile).  Run in the build container
(where /root/reference exists):   python tests/golden/make_golden.py

Inputs are not stored: tests/cases.py regenerates them deterministically.  Outputs are stored
in full (zip-compressed), keyed by case name, except where they are too large for the repository:
those are stored as sha256 digests (cases.digest), which the tests compare with the same digest of
what they computed.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))

import oracle  # noqa: E402
import cases  # noqa: E402
import timg_b200  # noqa: E402


def reference_random():
    """The reference's outputs on the random inputs of test_oracle_pinned.py / test_scale_oracle.py."""
    g = {}
    for seed in range(6):
        outs = cases.run_block_case(lambda *f: oracle.RefBlockCanvas(*f), cases.random_block_case(seed))
        for i, o in enumerate(outs):
            g[f"blocks_{seed}/{i}"] = np.frombuffer(o, np.uint8)
    for i, (fb, kw) in enumerate(cases.random_compose_cases()):
        g[f"compose_{i}"] = oracle.ref_compose_bg(fb, **kw)
    g["as256"] = np.array([oracle.ref().ref_as256(v) for v in cases.as256_values()], np.int16)
    g["scale"] = np.array([cases.digest(oracle.ref_scale(img, ow, oh, fmt))
                           for img, ow, oh, fmt in cases.random_scale_cases()])
    return g


def reference_configs():
    """Digests of the reference's outputs at BASELINE.json's config geometries (test_ref_gpu.py)."""
    bg = oracle.rgba_u32(0, 0, 0)
    g = {}
    for iw, ih, fit, kind in cases.CONFIG_GEOMETRIES:
        _, ow, oh = timg_b200.calc_fit(iw, ih, *fit)
        fb = oracle.ref_scale(cases.config_image(iw, ih, kind), ow, oh)
        g[f"scale_{iw}x{ih}_{ow}x{oh}"] = cases.digest(fb)
        g[f"compose_{iw}x{ih}_{ow}x{oh}"] = cases.digest(oracle.ref_compose_bg(fb, bg))
    frames = cases.c1_frames()
    _, ow, oh = timg_b200.calc_fit(640, 480, 80, 50, 1, 2)
    g["c1_half"] = np.array([cases.digest(oracle.RefBlockCanvas(False).send(
        oracle.ref_compose_bg(oracle.ref_scale(fr, ow, oh), bg))) for fr in frames])
    frames = cases.c3_frames()
    _, ow, oh = timg_b200.calc_fit(1920, 1080, 320, 100, 2, 2, 2.0)
    cv = oracle.RefBlockCanvas(True)
    g["c3_quarter_delta"] = np.array([cases.digest(cv.send(oracle.ref_compose_bg(oracle.ref_scale(fr, ow, oh), bg), 0,
                                                           0 if f == 0 else -oh)) for f, fr in enumerate(frames)])
    frames = cases.c4_frames()
    _, ow, oh = timg_b200.calc_fit(3840, 2160, 337, 225, 9, 18)
    hp = (oh + 5) // 6 * 6
    staged = []
    for fr in frames:                         # scale + compose, then SixelCanvas::Send's pad strip
        fb = np.zeros((hp, ow, 4), np.uint8)
        fb[:oh] = oracle.ref_compose_bg(oracle.ref_scale(fr, ow, oh), bg)
        staged.append(cases.digest(oracle.ref_compose_bg(fb, bg, start_row=oh)))
    g["c4_staged"] = np.array(staged)
    return g


def main():
    blocks = {}
    for name, case in cases.block_cases():
        outs = cases.run_block_case(lambda q, u, c: oracle.RefBlockCanvas(q, u, c), case)
        for i, o in enumerate(outs):
            blocks[f"{name}/{i}"] = np.frombuffer(o, np.uint8)
    np.savez_compressed(os.path.join(HERE, "blocks.npz"), **blocks)
    comp = {}
    for name, fb, kw in cases.compose_cases():
        comp[name] = oracle.ref_compose_bg(fb, **kw)
    np.savez_compressed(os.path.join(HERE, "compose.npz"), **comp)
    sc = {}
    for name, img, ow, oh, fmt in cases.scale_cases():
        sc[name] = oracle.ref_scale(img, ow, oh, fmt)
    np.savez_compressed(os.path.join(HERE, "scale.npz"), **sc)
    fit = []
    rng = np.random.default_rng(5)
    for _ in range(400):
        iw, ih = int(rng.integers(1, 5000)), int(rng.integers(1, 5000))
        width, height = int(rng.integers(1, 3000)), int(rng.integers(1, 3000))
        cx, cy = [(1, 2), (2, 2), (9, 18), (1, 1)][int(rng.integers(0, 4))]
        st = float(np.float32([1.0, 0.5, 2.0, 0.1, 7.0, 1.0, 0.8889][int(rng.integers(0, 7))]))
        fl = [int(v) for v in rng.integers(0, 2, 5)]
        args = (iw, ih, width, height, cx, cy, st, *fl)
        r = oracle.calc_fit(iw, ih, width, height, cx, cy, st, *map(bool, fl), impl=oracle.ref().ref_calc_fit)
        fit.append(list(args) + [int(r[0]), r[1], r[2]])
    np.savez_compressed(os.path.join(HERE, "fit.npz"), rows=np.array(fit, np.float64))
    np.savez_compressed(os.path.join(HERE, "reference_random.npz"), **reference_random())
    np.savez_compressed(os.path.join(HERE, "reference_configs.npz"), **reference_configs())
    total = sum(os.path.getsize(os.path.join(HERE, f)) for f in os.listdir(HERE) if f.endswith(".npz"))
    print(f"wrote {len(blocks)} block outputs, {len(comp)} compose outputs, {len(fit)} fit rows; {total} bytes")


if __name__ == "__main__":
    main()

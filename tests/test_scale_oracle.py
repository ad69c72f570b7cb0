"""Pins the scaler restatement (oracle/stbir_oracle.c) against the golden outputs produced by
the reference's own STB scaler, and the product's host-side resampling plan against the
oracle's.  No GPU needed."""
import os

import numpy as np

import cases
import oracle
import timg_b200

G = os.path.join(os.path.dirname(__file__), "golden")


def test_scale_oracle_matches_golden():
    g = np.load(os.path.join(G, "scale.npz"))
    for name, img, ow, oh, fmt in cases.scale_cases():
        assert (oracle.stb_resize(img, ow, oh, fmt) == g[name]).all(), name


def test_identity_is_exact_copy():
    v = np.arange(256, dtype=np.uint8)
    img = np.stack(np.meshgrid(v, v), -1)
    img = np.concatenate([img, img[..., ::-1]], -1)          # every byte value in every channel
    assert (oracle.stb_resize(img, 256, 256) == img).all()


def _plans_equal(a, b):
    return (a["widest"] == b["widest"] and a["flags"] == b["flags"]
            and all((a[k] == b[k]).all() for k in ("first", "count", "lead"))
            and (a["coeff"].view(np.uint32) == b["coeff"].view(np.uint32)).all())


def test_product_plan_equals_oracle_plan_on_config_geometries():
    for iw, ih, ow, oh in [(640, 480, 67, 50), (3840, 2160, 2700, 1519), (1920, 1080, 320, 90),
                           (3840, 2160, 337, 190), (1280, 720, 1280, 720), (3840, 2160, 600, 168)]:
        for ax in (0, 1):
            assert _plans_equal(timg_b200.resample_plan(iw, ih, ow, oh, ax), oracle.stb_plan(iw, ih, ow, oh, ax))


def test_product_plan_equals_oracle_plan_random():
    rng = np.random.default_rng(4)
    for it in range(150):
        iw, ih = int(rng.integers(1, 2000)), int(rng.integers(1, 1500))
        m = it % 4
        if m == 0:
            ow, oh = int(rng.integers(1, 2000)), int(rng.integers(1, 1500))
        elif m == 1:
            ow, oh = max(1, iw // int(rng.integers(1, 40))), max(1, ih // int(rng.integers(1, 40)))
        elif m == 2:
            ow, oh = iw * int(rng.integers(1, 4)), ih * int(rng.integers(1, 4))
        else:
            ow, oh = iw, int(rng.integers(1, 1500))
        for ax in (0, 1):
            assert _plans_equal(timg_b200.resample_plan(iw, ih, ow, oh, ax), oracle.stb_plan(iw, ih, ow, oh, ax)), \
                (iw, ih, ow, oh, ax)


def test_c2_plan_shape():
    """4K -> 2700x1519 (BASELINE config 1): 45/64 polyphase horizontally, 6 taps per axis."""
    h = timg_b200.resample_plan(3840, 2160, 2700, 1519, 0)
    v = timg_b200.resample_plan(3840, 2160, 2700, 1519, 1)
    assert h["widest"] == 6 and v["widest"] == 6
    assert (h["first"][47:90] - h["first"][2:45] == 64).all()     # period 45 out / 64 in (edge-clamped at 0,1)
    np.testing.assert_allclose(h["coeff"].sum(1), 1.0, atol=1e-6)
    np.testing.assert_allclose(v["coeff"].sum(1), 1.0, atol=1e-6)


def test_scale_oracle_vs_reference_random():
    """The reference's outputs on these inputs are stored as digests (they would not fit the repository)."""
    want = np.load(os.path.join(G, "reference_random.npz"))["scale"]
    for (img, ow, oh, fmt), d in zip(cases.random_scale_cases(), want, strict=True):
        assert cases.digest(oracle.stb_resize(img, ow, oh, fmt)) == d, (img.shape, ow, oh, fmt)

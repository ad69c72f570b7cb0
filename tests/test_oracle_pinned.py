"""Pins the CPU oracle (oracle/*.c, our restatement) against the golden fixtures generated from the
reference itself (tests/golden/*.npz, written by tests/golden/make_golden.py): fixed cases and random
inputs.  No GPU needed."""
import os

import numpy as np
import pytest

import cases
import oracle

G = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def golden_blocks():
    return np.load(os.path.join(G, "blocks.npz"))


@pytest.fixture(scope="module")
def golden_random():
    return np.load(os.path.join(G, "reference_random.npz"))


@pytest.mark.parametrize("name,case", cases.block_cases(), ids=[n for n, _ in cases.block_cases()])
def test_blocks_oracle_matches_golden(name, case, golden_blocks):
    outs = cases.run_block_case(lambda q, u, c: oracle.BlockCanvas(q, u, c), case)
    for i, o in enumerate(outs):
        assert o == golden_blocks[f"{name}/{i}"].tobytes(), f"{name} frame {i}"


def test_appendix_d_bytes(golden_blocks):
    """The worked delta example of SURVEY.md App. D, spelled out."""
    g = lambda i: golden_blocks[f"delta_appD_q0u0/{i}"].tobytes()
    assert g(0) == 8 * b"\033[48;2;10;20;30m    \033[0m\n"
    assert g(1) == b"\033[8A\033[6B\033[2C\033[38;2;200;100;50;48;2;10;20;30m\xe2\x96\x84\033[0m\n\033[1B"
    assert g(2) == b""
    assert g(3) == (b"\033[8A\n\033[38;2;10;20;30;48;2;1;2;3m\xe2\x96\x84\033[2C"
                    b"\033[38;2;1;2;3;48;2;10;20;30m\xe2\x96\x84\033[0m\n\033[6B")


def test_compose_oracle_matches_golden():
    g = np.load(os.path.join(G, "compose.npz"))
    for name, fb, kw in cases.compose_cases():
        assert (oracle.compose_bg(fb, **kw) == g[name]).all(), name


def test_fit_oracle_and_product_match_golden():
    import timg_b200
    rows = np.load(os.path.join(G, "fit.npz"))["rows"]
    for row in rows:
        iw, ih, width, height, cx, cy = (int(v) for v in row[:6])
        st = float(np.float32(row[6]))
        up, upi, fw, fh, rot = (bool(v) for v in row[7:12])
        want = (bool(row[12]), int(row[13]), int(row[14]))
        assert oracle.calc_fit(iw, ih, width, height, cx, cy, st, up, upi, fw, fh, rot) == want
        assert timg_b200.calc_fit(iw, ih, width, height, cx, cy, st, up, upi, fw, fh, rot) == want


def test_config_geometries():
    """The scaled-framebuffer sizes SURVEY.md 8(d) quotes for BASELINE.json's configs."""
    import timg_b200
    for fit in (oracle.calc_fit, timg_b200.calc_fit):
        assert fit(640, 480, 80, 50, 1, 2)[1:] == (67, 50)                       # C1 -p half -g80x25
        assert fit(3840, 2160, 2700, 1800, 9, 18)[1:] == (2700, 1519)           # C2 -p sixel -g300x100
        assert fit(1920, 1080, 320, 100, 2, 2, 2.0)[1:] == (320, 90)            # C3 -p quarter -g160x50 (width_stretch*=2, src/timg.cc:838)
        assert fit(3840, 2160, 337, 225, 9, 18)[1:] == (337, 190)               # C4 --grid=8x8
        assert fit(1280, 720, 2700, 1800, 9, 18) == (False, 1280, 720)          # C5 no upscale


def test_as256_all_colours(golden_random):
    import timg_b200
    vals = cases.as256_values()
    got_o = [oracle.as256(v) for v in vals]
    got_p = [timg_b200.lib().b200timg_as256(v) for v in vals]
    assert got_o == got_p
    assert got_o == golden_random["as256"].tolist()


@pytest.mark.parametrize("seed", range(6))
def test_blocks_oracle_vs_reference_random(seed, golden_random):
    outs = cases.run_block_case(lambda *f: oracle.BlockCanvas(*f), cases.random_block_case(seed))
    for i, o in enumerate(outs):
        assert o == golden_random[f"blocks_{seed}/{i}"].tobytes(), f"frame {i}"


def test_compose_oracle_vs_reference_random(golden_random):
    for i, (fb, kw) in enumerate(cases.random_compose_cases()):
        assert (oracle.compose_bg(fb, **kw) == golden_random[f"compose_{i}"]).all(), i

"""Pin the oracle's reduced-size IDCTs (decodes at 1/2, 1/4, 1/8 scale) against libjpeg-turbo before the GPU is compared
with them (test_scaled_gpu.py).

libjpeg-turbo transforms every component at scale 1/d with the reduced IDCT of jidctred.c of size 8/d, except 4:2:0
chroma, which it decodes with the next larger transform (16/d) to save upsampling. The decoder keeps the coded chroma
ratio and uses 8/d for every component, so:
  - every component libjpeg-turbo transforms at 8/d must equal it bit for bit;
  - 4:2:0 chroma at 1/2 and 1/4 is checked against libjpeg-turbo's chroma at 1/4 and 1/8, where it uses exactly that
    transform size; 4:2:0 chroma at 1/8 is the 1x1 transform, which every other fixture's components pin.
"""
import json
import os

import numpy as np
import pytest

import oracle
import scaled_oracle as so

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden")
with open(os.path.join(GOLDEN, "golden.json")) as _f:
    CASES = sorted(json.load(_f)["cases"])
SCALES = (2, 4, 8)


@pytest.fixture(scope="module")
def sorc(orc):
    return so.ScaledOracle(orc)


@pytest.fixture(scope="module")
def sljt():
    return so.ScaledLibJpegTurbo()


def load(name):
    with open(os.path.join(GOLDEN, name + ".jpg"), "rb") as f:
        return f.read()


def test_libjpeg_turbo_offsets_for_scaled_decodes(sljt):
    """The cinfo fields the scaled harness writes and reads (scale_num / scale_denom, output size, DCT_scaled_size)."""
    for name in ("synth_444_123x77", "synth_420_123x77", "synth_400_333x211"):
        assert sljt.selfcheck(load(name)) == 0, name


@pytest.mark.parametrize("d", SCALES)
@pytest.mark.parametrize("name", CASES)
def test_scaled_planes_match_libjpeg_turbo(orc, sorc, ljt, sljt, name, d):
    data = load(name)
    rc, info = orc.parse(data)
    assert rc == 0
    sinfo = so.scaled_info(info, d)
    assert (sinfo.width, sinfo.height) == sljt.output_size(data, d), "ceil(W/d) x ceil(H/d)"
    planes = sorc.planes_scaled(data, d, info)
    lp, dss = sljt.raw_planes_scaled(data, info, d)
    li = ljt.info(data)
    s = 8 // d
    for c in range(info.ncomp):
        assert planes[c].shape == (info.blocks_h[c] * s, info.blocks_w[c] * s)
        if dss[c] == s:
            want = lp[c]
        else:
            # 4:2:0 chroma: libjpeg-turbo's transform of that size is the one of its decode at half this scale
            assert oracle.CSS[info.css] == "420" and c > 0 and dss[c] == 2 * s, (dss, c)
            if d == 8:
                continue
            lp2, dss2 = sljt.raw_planes_scaled(data, info, 2 * d)
            assert dss2[c] == s
            want = lp2[c]
        hh, ww = li.hib[c] * s, li.wib[c] * s   # libjpeg does not transform the dummy blocks beyond these
        assert np.array_equal(planes[c][:hh, :ww], want[:hh, :ww]), f"component {c} at 1/{d}"


@pytest.mark.parametrize("name", CASES)
def test_scale_one_is_the_islow_path(orc, sorc, name):
    data = load(name)
    rc, info = orc.parse(data)
    full = orc.planes(data, info)
    one = sorc.planes_scaled(data, 1, info)
    for c in range(info.ncomp):
        assert np.array_equal(one[c], full[c])
    _, a = orc.decode(data, "rgb")
    _, b = sorc.decode_scaled(data, 1, "rgb")
    assert all(np.array_equal(x, y) for x, y in zip(a, b))


def test_scaled_block_closed_forms(sorc):
    """DC-only blocks: every transform size yields a flat block of (DC*q + 4) >> 3, +128, saturated."""
    q = np.ones(64, dtype=np.uint16) * 3
    for dc in (-400, -43, -1, 0, 1, 17, 42, 300):
        coef = np.zeros(64, dtype=np.int16)
        coef[0] = dc
        want = min(255, max(0, ((dc * 3 + 4) >> 3) + 128))
        for d in (1, 2, 4, 8):
            s = 8 // d
            out = sorc.idct_block(coef, q, d)
            assert out.shape == (s, s) and (out == want).all(), (dc, d)

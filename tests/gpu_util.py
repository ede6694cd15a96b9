"""Helpers for the -m gpu parity tests: decode through the C ABI into torch-owned device
buffers with chosen pitches / base misalignment, return host copies of the WHOLE buffers
(so stray writes outside the valid region are visible)."""
import numpy as np

import oracle
from rocjpeg_b200 import api

FILL = 0xCD


def roi_dims(orc, info, crop):
    rc, x0, y0, w, h = orc.roi(info, crop)
    return rc, w, h


def output_layout(orc, info, fmt, crop, pitch_pad=0):
    """(shapes, pitches) of the destination channels of one picture: (rows, valid bytes per row) and the pitch of each."""
    shapes = oracle.output_shapes(info, fmt, crop, orc)
    pitches = [rb + pitch_pad for (_, rb) in shapes]
    css = oracle.CSS[info.css]
    if fmt == "yuv_planar" and css in ("422", "420") and len(pitches) == 3:
        pitches[2] = pitches[1]          # U and V share pitch[1] (src/rocjpeg_decoder.cpp:589-597)
    if fmt == "rgb_planar":
        pitches[1] = pitches[2] = pitches[0]
    return shapes, pitches


def alloc_outputs(orc, info, fmt, crop, pitch_pad=0, misalign=0):
    """Returns (dest list for api.Decoder, torch buffers, pitches, shapes)."""
    import torch

    shapes, pitches = output_layout(orc, info, fmt, crop, pitch_pad)
    bufs, dest = [], []
    for (rows, _), p in zip(shapes, pitches):
        t = torch.full((rows * p + misalign + 64,), FILL, dtype=torch.uint8, device="cuda")
        bufs.append(t)
        dest.append((t.data_ptr() + misalign, p))
    return dest, bufs, pitches, shapes


def fetch(bufs, pitches, shapes, misalign=0):
    out = []
    for t, p, (rows, _) in zip(bufs, pitches, shapes):
        a = t.cpu().numpy()
        assert (a[:misalign] == FILL).all() and (a[misalign + rows * p:] == FILL).all(), "write outside the channel buffer"
        out.append(a[misalign:misalign + rows * p].reshape(rows, p))
    return out


def oracle_outputs(orc, data, fmt, crop, pitches):
    info, dst = orc.decode(data, fmt, crop, pitches=pitches, fill=FILL)
    return info, dst


def decode_one(dec, orc, data, fmt, crop=(0, 0, 0, 0), pitch_pad=0, misalign=0):
    """Decode one image with rocJpegDecode; returns (status, got arrays, oracle arrays)."""
    s = api.JpegStream()
    st = s.parse(data)
    assert st == api.SUCCESS, st
    rc, info = orc.parse(data)
    dest, bufs, pitches, shapes = alloc_outputs(orc, info, fmt, crop, pitch_pad, misalign)
    st = dec.decode(s, api.make_params(fmt, crop), dest)
    if st != api.SUCCESS:
        return st, None, None
    got = fetch(bufs, pitches, shapes, misalign)
    _, want = oracle_outputs(orc, data, fmt, crop, pitches)
    return st, got, want


def assert_same(got, want, what=""):
    assert len(got) == len(want), what
    for c, (g, w) in enumerate(zip(got, want)):
        assert g.shape == w.shape, (what, c, g.shape, w.shape)
        if not np.array_equal(g, w):
            bad = np.argwhere(g != w)
            raise AssertionError(f"{what}: channel {c}: {len(bad)} bytes differ, first at {bad[0].tolist()} "
                                 f"got {g[tuple(bad[0])]} want {w[tuple(bad[0])]}")

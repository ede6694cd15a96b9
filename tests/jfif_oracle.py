"""CPU restatement of RGB under the libjpeg colour convention - TEST INFRASTRUCTURE ONLY (tests/ and profiles/bench_color.py).

tests/jfif_oracle.c (fancy chroma upsampling + JFIF integer colour, libjpeg-turbo's jdsample.c / jdcolor.c) is compiled
together with the unchanged oracle source it includes into a library of its own on first use, under tests/_build/ - or a
temporary directory when the tree is read-only - as tests/scaled_oracle.py does. It runs on the oracle's planes: full size,
or the reduced-size planes of scaled_oracle.ScaledOracle.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

import oracle
import scaled_oracle as so

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_DIR = os.path.join(os.path.dirname(HERE), "oracle")


def _library() -> str:
    srcs = [os.path.join(HERE, "jfif_oracle.c"), os.path.join(ORACLE_DIR, "jpeg_oracle.c")]
    out = os.path.join(so._build_dir(), "libjfif_oracle.so")
    if not os.path.exists(out) or any(os.path.getmtime(s) > os.path.getmtime(out) for s in srcs):
        tmp = f"{out}.{os.getpid()}.tmp"
        r = subprocess.run(["gcc", "-O2", "-shared", "-fPIC", "-I", ORACLE_DIR, "-o", tmp, srcs[0], "-lm"],
                           capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"building libjfif_oracle.so failed:\n{r.stdout}{r.stderr}")
        os.replace(tmp, out)
    return out


class JfifOracle:
    """RGB / RGB_PLANAR as libjpeg-turbo's default decode makes them, from the oracle's planes at scale 1/d, assembled with
    the oracle's crop and pitch rules."""

    def __init__(self, orc: oracle.Oracle | None = None):
        self.orc = orc or oracle.Oracle()
        self.scaled = so.ScaledOracle(self.orc)
        self.lib = C.CDLL(_library())
        self.lib.orc_info_size.restype = C.c_size_t
        assert self.lib.orc_info_size() == C.sizeof(oracle.OrcInfo)
        self.lib.jfif_convert.argtypes = [C.POINTER(oracle.OrcInfo), C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]

    def planes(self, data: bytes, info, d: int) -> list[np.ndarray]:
        """The planes in orc_idct_planes' layout at scale 1/d."""
        if d == 1:
            return self.orc.planes(data, info)
        return self.scaled.planes_scaled_full(info, self.orc.coefficients(data, info), d)

    def decode(self, data: bytes, fmt: str, d: int = 1, crop=(0, 0, 0, 0), pitches=None, fill=0xCD):
        """Returns (info at the output size, [channel arrays shaped (rows, pitch)]); `crop` is in output coordinates."""
        rc, info = self.orc.parse(data)
        if rc != 0:
            raise ValueError(f"parse rc={rc}")
        planes = self.planes(data, info, d)
        sinfo = so.scaled_info(info, d)
        shapes = oracle.output_shapes(sinfo, fmt, crop, self.orc)
        dst, pit = [], []
        for i, (rows, rowbytes) in enumerate(shapes):
            p = rowbytes if pitches is None else pitches[i]
            pit.append(p)
            dst.append(np.full((rows, p), fill, dtype=np.uint8))
        flat = np.ascontiguousarray(np.concatenate([p.reshape(-1) for p in planes]))
        c = np.array(crop, dtype=np.int16)
        ptrs = (C.c_void_p * 4)(*[a.ctypes.data for a in dst] + [None] * (4 - len(dst)))
        pa = (C.c_uint32 * 4)(*(pit + [0] * (4 - len(pit))))
        rc = self.lib.jfif_convert(C.byref(sinfo), flat.ctypes.data, d, oracle.FMT[fmt], c.ctypes.data, ptrs, pa)
        if rc != 0:
            raise ValueError(f"jfif_convert rc={rc}")
        return sinfo, dst

    def rgb(self, data: bytes, d: int = 1) -> np.ndarray:
        """The whole picture at scale 1/d as (H, W, 3) RGB."""
        sinfo, dst = self.decode(data, "rgb", d)
        return dst[0].reshape(sinfo.height, sinfo.width, 3)

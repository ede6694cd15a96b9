"""CPU oracle for decodes at 1/2, 1/4 and 1/8 scale - TEST INFRASTRUCTURE ONLY (tests/ and profiles/bench_scaled.py).

Extends the oracle package without changing it: tests/scaled_oracle.c (the reduced-size IDCTs of libjpeg's jidctred.c)
and tests/ljt_scaled.c (libjpeg-turbo at scale_denom 2, 4, 8) are each compiled together with the unchanged oracle
source they include (oracle/jpeg_oracle.c, oracle/ljt_shim.c) into a library of their own, on first use, under
tests/_build/ - or a temporary directory when the tree is read-only.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

import oracle

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_DIR = os.path.join(os.path.dirname(HERE), "oracle")
_LIBS = {
    "libscaled_oracle.so": (["scaled_oracle.c", "jpeg_oracle.c"], ["-O2", "-ffp-contract=off", "-fno-fast-math"], ["-lm"]),
    "libljt_scaled.so": (["ljt_scaled.c", "ljt_shim.c"], ["-O2"], ["-ldl", "-lpthread"]),
}


def _build_dir():
    d = os.path.join(HERE, "_build")
    try:
        os.makedirs(d, exist_ok=True)
        if os.access(d, os.W_OK):
            return d
    except OSError:
        pass
    d = os.path.join(tempfile.gettempdir(), f"rocjpeg_b200_scaled_oracle_{os.getuid()}")
    os.makedirs(d, exist_ok=True)
    return d


def _library(name: str) -> str:
    (src, *deps), cflags, libs = _LIBS[name]
    srcs = [os.path.join(HERE, src)] + [os.path.join(ORACLE_DIR, x) for x in deps]
    out = os.path.join(_build_dir(), name)
    if not os.path.exists(out) or any(os.path.getmtime(s) > os.path.getmtime(out) for s in srcs):
        tmp = f"{out}.{os.getpid()}.tmp"
        r = subprocess.run(["gcc", *cflags, "-shared", "-fPIC", "-I", ORACLE_DIR, "-o", tmp, srcs[0], *libs],
                           capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"building {name} failed:\n{r.stdout}{r.stderr}")
        os.replace(tmp, out)
    return out


def scaled_info(info, d: int):
    """Copy of an OrcInfo with width / height at scale 1/d: ceil(W/d) x ceil(H/d) (libjpeg's output_width / height)."""
    s = oracle.OrcInfo()
    C.pointer(s)[0] = info
    s.width, s.height = -(-info.width // d), -(-info.height // d)
    return s


class ScaledOracle:
    """The oracle's path at scale 1/d: reduced-size IDCT of the oracle's coefficients, then its output assembly
    (orc_convert) at the scaled size. Parsing, coefficients and assembly are the wrapped oracle.Oracle's."""

    def __init__(self, orc: oracle.Oracle | None = None):
        self.orc = orc or oracle.Oracle()
        self.lib = C.CDLL(_library("libscaled_oracle.so"))
        self.lib.orc_info_size.restype = C.c_size_t
        assert self.lib.orc_info_size() == C.sizeof(oracle.OrcInfo)
        self.lib.orc_idct_scaled_block.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int]
        self.lib.orc_idct_planes_scaled.argtypes = [C.POINTER(oracle.OrcInfo), C.c_void_p, C.c_int, C.c_void_p]

    scaled_info = staticmethod(scaled_info)

    def idct_block(self, coef_nat, q_nat, d: int) -> np.ndarray:
        """One block at scale 1/d: (8/d) x (8/d) samples."""
        coef = np.ascontiguousarray(coef_nat, dtype=np.int16).reshape(64)
        q = np.ascontiguousarray(q_nat, dtype=np.uint16).reshape(64)
        out = np.zeros((8, 8), dtype=np.uint8)
        self.lib.orc_idct_scaled_block(coef.ctypes.data, q.ctypes.data, d, out.ctypes.data, 8)
        return out[:8 // d, :8 // d].copy()

    def planes_scaled_full(self, info, coefs, d: int) -> list[np.ndarray]:
        """Planes at scale 1/d from per-component coefficient arrays, in orc_idct_planes_scaled's layout: per component
        a (blocks_h*8, blocks_w*8) array whose top-left (blocks_h*8/d, blocks_w*8/d) corner holds the scaled plane."""
        flat_c = np.ascontiguousarray(np.concatenate([c.reshape(-1) for c in coefs]), dtype=np.int16)
        flat = np.zeros(flat_c.size, dtype=np.uint8)
        rc = self.lib.orc_idct_planes_scaled(C.byref(info), flat_c.ctypes.data, d, flat.ctypes.data)
        if rc != 0:
            raise ValueError(f"orc_idct_planes_scaled rc={rc}")
        out, base = [], 0
        for c in range(info.ncomp):
            bw, bh = info.blocks_w[c], info.blocks_h[c]
            out.append(flat[base:base + bw * bh * 64].reshape(bh * 8, bw * 8))
            base += bw * bh * 64
        return out

    def planes_scaled(self, data: bytes, d: int, info=None, coefs=None) -> list[np.ndarray]:
        """Per component: uint8 plane (blocks_h*8/d, blocks_w*8/d) decoded with the reduced-size IDCT of scale 1/d
        (the layout rocJpegB200GetPlanes returns after a scaled decode). `coefs` (optional) replaces the stream's."""
        if info is None:
            rc, info = self.orc.parse(data)
            assert rc == 0, rc
        if coefs is None:
            coefs = self.orc.coefficients(data, info)
        full = self.planes_scaled_full(info, coefs, d)
        s = 8 // d
        return [np.ascontiguousarray(p[:info.blocks_h[c] * s, :info.blocks_w[c] * s]) for c, p in enumerate(full)]

    def decode_scaled(self, data: bytes, d: int, fmt: str, crop=(0, 0, 0, 0), pitches=None, fill=0xCD):
        """Oracle.decode at scale 1/d: the output assembly of the scaled planes at the scaled size; `crop` is in scaled
        coordinates. Returns (scaled info, [channel arrays shaped (rows, pitch)], None for a channel with no rows)."""
        rc, info = self.orc.parse(data)
        if rc != 0:
            raise ValueError(f"parse rc={rc}")
        rc = self.orc.supported(info)
        if rc != 0:
            raise ValueError(f"unsupported rc={rc}")
        planes = self.planes_scaled_full(info, self.orc.coefficients(data, info), d)
        sinfo = scaled_info(info, d)
        shapes = oracle.output_shapes(sinfo, fmt, crop, self.orc)
        dst, pit = [], []
        for i, (rows, rowbytes) in enumerate(shapes):
            p = rowbytes if pitches is None else pitches[i]
            pit.append(p)
            dst.append(np.full((rows, p), fill, dtype=np.uint8) if rows and p else None)
        rc = self.orc.convert(sinfo, planes, fmt, crop, dst, pit)
        if rc != 0:
            raise ValueError(f"convert rc={rc}")
        return sinfo, dst


class ScaledLibJpegTurbo:
    """Pillow's bundled libjpeg-turbo at scale_num 1, scale_denom d."""

    def __init__(self):
        self.lib = C.CDLL(_library("libljt_scaled.so"))
        self.path = oracle.find_libjpeg_turbo()
        rc = self.lib.ljt_open(self.path.encode())
        if rc != 0:
            raise RuntimeError(f"ljt_open({self.path}) rc={rc}")
        L = self.lib
        L.ljt_read_raw_scaled.argtypes = [C.c_void_p, C.c_size_t, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.ljt_output_size.argtypes = [C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]
        L.ljt_selfcheck.argtypes = [C.c_void_p, C.c_size_t]
        L.ljt_decode_batch_scaled.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]

    def selfcheck(self, data: bytes) -> int:
        """0 when the struct offsets the scaled decodes use hold on this stream."""
        return self.lib.ljt_selfcheck(data, len(data))

    def output_size(self, data: bytes, d: int) -> tuple[int, int]:
        """(output_width, output_height) libjpeg-turbo decodes the stream to at scale 1/d."""
        wh = (C.c_int32 * 2)()
        rc = self.lib.ljt_output_size(data, len(data), d, wh)
        if rc:
            raise ValueError(f"ljt_output_size rc={rc}")
        return wh[0], wh[1]

    def raw_planes_scaled(self, data: bytes, oinfo, d: int):
        """jpeg_read_raw_data at scale 1/d. Returns (planes, dss): per component the (bh*dss, bw*dss) plane libjpeg-turbo
        produced with its DCT_scaled_size dss[c] (8/d, except 4:2:0 chroma: 16/d)."""
        bw = (C.c_int32 * 3)(*oinfo.blocks_w)
        bh = (C.c_int32 * 3)(*oinfo.blocks_h)
        dss = (C.c_int32 * 3)()
        n = sum(oinfo.blocks_w[c] * oinfo.blocks_h[c] * 64 for c in range(oinfo.ncomp))
        flat = np.zeros(n, dtype=np.uint8)
        rc = self.lib.ljt_read_raw_scaled(data, len(data), d, flat.ctypes.data, bw, bh, dss)
        if rc:
            raise ValueError(f"ljt_read_raw_scaled rc={rc}")
        out, base = [], 0
        for c in range(oinfo.ncomp):
            w, h = oinfo.blocks_w[c] * 8, oinfo.blocks_h[c] * 8
            full = flat[base:base + w * h].reshape(h, w)
            out.append(np.ascontiguousarray(full[:oinfo.blocks_h[c] * dss[c], :oinfo.blocks_w[c] * dss[c]]))
            base += w * h
        return out, list(dss)[:oinfo.ncomp]

    def decode_batch_scaled(self, datas: list[bytes], outs: list[np.ndarray], pitches: list[int], mode: int, nthreads: int,
                            d: int):
        """Multithreaded decode at scale 1/d (mode 0: ceil(W/d) x ceil(H/d) RGB pixels, 2: raw planes); releases the GIL."""
        n = len(datas)
        dptr = (C.c_char_p * n)(*datas)
        lens = (C.c_size_t * n)(*[len(x) for x in datas])
        optr = (C.c_void_p * n)(*[o.ctypes.data for o in outs])
        pit = (C.c_size_t * n)(*pitches)
        rc = self.lib.ljt_decode_batch_scaled(n, dptr, lens, optr, pit, mode, nthreads, d)
        if rc:
            raise ValueError(f"ljt_decode_batch_scaled rc={rc}")

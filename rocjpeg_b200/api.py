"""ctypes binding of rocjpeg_b200/lib/librocjpeg.so — the same nine entry points a
C/C++ caller of the reference binds (api/rocjpeg.h:204-343), plus the rocJpegB200*
extension taps (include/rocjpeg_b200_ext.h).

The reference is a C++ library, so the product's host side is C++ (csrc/); this
module is only the Python-visible mirror used by tests/ and bench.py. There is no
CPU fallback: without the built CUDA library every call here raises.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("ROCJPEG_B200_LIB") or os.path.join(HERE, "lib", "librocjpeg.so")   # the override serves debugging builds

# RocJpegStatus (include/rocjpeg.h, api/rocjpeg.h:53-67)
STATUS = {
    0: "ROCJPEG_STATUS_SUCCESS", -1: "ROCJPEG_STATUS_NOT_INITIALIZED", -2: "ROCJPEG_STATUS_INVALID_PARAMETER",
    -3: "ROCJPEG_STATUS_BAD_JPEG", -4: "ROCJPEG_STATUS_JPEG_NOT_SUPPORTED", -5: "ROCJPEG_STATUS_OUTOF_MEMORY",
    -6: "ROCJPEG_STATUS_EXECUTION_FAILED", -7: "ROCJPEG_STATUS_ARCH_MISMATCH", -8: "ROCJPEG_STATUS_INTERNAL_ERROR",
    -9: "ROCJPEG_STATUS_IMPLEMENTATION_NOT_SUPPORTED", -10: "ROCJPEG_STATUS_HW_JPEG_DECODER_NOT_SUPPORTED",
    -11: "ROCJPEG_STATUS_RUNTIME_ERROR", -12: "ROCJPEG_STATUS_NOT_IMPLEMENTED",
}
SUCCESS, NOT_INITIALIZED, INVALID_PARAMETER, BAD_JPEG, JPEG_NOT_SUPPORTED = 0, -1, -2, -3, -4
EXECUTION_FAILED, RUNTIME_ERROR, NOT_IMPLEMENTED = -6, -11, -12
# RocJpegChromaSubsampling (api/rocjpeg.h:86-94)
CSS_444, CSS_440, CSS_422, CSS_420, CSS_411, CSS_400, CSS_UNKNOWN = 0, 1, 2, 3, 4, 5, -1
CSS_NAME = {0: "444", 1: "440", 2: "422", 3: "420", 4: "411", 5: "400", -1: "unknown"}
# RocJpegOutputFormat (api/rocjpeg.h:124-141)
OUTPUT_NATIVE, OUTPUT_YUV_PLANAR, OUTPUT_Y, OUTPUT_RGB, OUTPUT_RGB_PLANAR = 0, 1, 2, 3, 4
FMT = {"native": 0, "yuv_planar": 1, "y": 2, "rgb": 3, "rgb_planar": 4}
# RocJpegBackend (api/rocjpeg.h:176-179)
BACKEND_HARDWARE, BACKEND_HYBRID = 0, 1
STAGES = ("upload", "destuff", "huffman_sync", "huffman_write", "dc", "idct", "output")


class RocJpegImage(C.Structure):
    _fields_ = [("channel", C.c_void_p * 4), ("pitch", C.c_uint32 * 4)]


class _Crop(C.Structure):
    _fields_ = [("left", C.c_int16), ("top", C.c_int16), ("right", C.c_int16), ("bottom", C.c_int16)]


class _Target(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32)]


class RocJpegDecodeParams(C.Structure):
    _fields_ = [("output_format", C.c_int), ("crop_rectangle", _Crop), ("target_dimension", _Target)]


class Stats(C.Structure):
    _fields_ = [
        ("stage_ms", C.c_float * 7), ("total_ms", C.c_float), ("sync_rounds", C.c_uint32),
        ("decodes_per_round", C.c_uint32 * 8), ("scan_bytes", C.c_uint64), ("blocks", C.c_uint64),
        ("subsequences", C.c_uint64), ("plane_bytes", C.c_uint64), ("output_bytes", C.c_uint64),
        ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64), ("kernel_launches", C.c_uint32),
        ("subsequence_bytes", C.c_int32), ("lanes", C.c_int32),
        ("host_submit_ms", C.c_float), ("host_wait_ms", C.c_float), ("devices", C.c_int32),
        ("entries", C.c_uint64), ("truncated_images", C.c_uint32), ("pad_", C.c_uint32), ("fused_blocks", C.c_uint64),
    ]


class StreamInfo(C.Structure):
    _fields_ = [
        ("width", C.c_int32), ("height", C.c_int32), ("num_components", C.c_int32), ("chroma_subsampling", C.c_int32),
        ("h_sampling", C.c_int32 * 3), ("v_sampling", C.c_int32 * 3), ("quant_selector", C.c_int32 * 3),
        ("dc_selector", C.c_int32 * 3), ("ac_selector", C.c_int32 * 3), ("restart_interval", C.c_int32),
        ("num_mcus", C.c_uint32), ("scan_offset", C.c_uint32), ("raw_bytes", C.c_uint32),
        ("mcus_x", C.c_int32), ("mcus_y", C.c_int32), ("blocks_per_mcu", C.c_int32),
        ("blocks_w", C.c_int32 * 3), ("blocks_h", C.c_int32 * 3), ("num_segments", C.c_uint32),
        ("decode_status", C.c_int32), ("source_is_device_visible", C.c_int32), ("source_is_zero_copy", C.c_int32),
        ("features", C.c_int32),
    ]


class ScanStatus(C.Structure):
    _fields_ = [("segments_seen", C.c_uint32), ("scan_size", C.c_uint32), ("flags", C.c_uint32), ("reserved", C.c_uint32)]


FEAT_SOF1, FEAT_DQT16, FEAT_HUFF_ID23 = 1, 2, 4
SCAN_NO_EOI, SCAN_STRAY_MARKER, SCAN_EXTRA_RESTARTS, SCAN_MISSING_INTERVALS, SCAN_EMPTY_INTERVAL = 1, 2, 4, 8, 16
DECODE_SHORT, TRUNCATED_MASK = 32, 8 | 16 | 32


class HostScanInfo(C.Structure):
    _fields_ = [("scan_size", C.c_uint32), ("restart_markers_seen", C.c_uint32), ("num_segments", C.c_uint32),
                ("clean_bytes", C.c_uint64)]


EXPORTS = (
    "rocJpegStreamCreate", "rocJpegStreamParse", "rocJpegStreamDestroy", "rocJpegCreate", "rocJpegDestroy",
    "rocJpegGetImageInfo", "rocJpegDecode", "rocJpegDecodeBatched", "rocJpegGetErrorName",
)
EXT_EXPORTS = (
    "rocJpegB200SetProfiling", "rocJpegB200GetStats", "rocJpegB200Prepare", "rocJpegB200Run",
    "rocJpegB200GetCoefficients", "rocJpegB200GetPlanes", "rocJpegB200StreamGetInfo", "rocJpegB200StreamGetSegment",
    "rocJpegB200StreamGetQuantTable", "rocJpegB200StreamGetHuffmanTable", "rocJpegB200Version", "rocJpegB200StreamGetLastError",
    "rocJpegB200PlanShards", "rocJpegB200GetDeviceCount", "rocJpegB200StreamHostScan",
    "rocJpegB200GetScanStatus", "rocJpegB200GetDeviceSegment", "rocJpegB200ParseAndDecodeBatched",
    "rocJpegB200PlanShardsPinned", "rocJpegB200GetImageStatus", "rocJpegB200StreamLoadFiles",
    "rocJpegB200GetScaledImageInfo", "rocJpegB200DecodeBatchedScaled", "rocJpegB200PrepareScaled",
)
SCALES = (1, 2, 4, 8)   # denominators of the reduced-size decodes

_lib = None


class RocJpegError(RuntimeError):
    def __init__(self, status: int, where: str):
        self.status = status
        super().__init__(f"{where}: {STATUS.get(status, status)}")


def load_library() -> C.CDLL:
    """Load the CUDA decoder library; fails loudly if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `make -C rocjpeg_b200/csrc` (or __graft_entry__.build()). "
            "rocjpeg_b200 has no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, i32 = C.c_void_p, C.c_int
    L.rocJpegStreamCreate.argtypes = [C.POINTER(vp)]
    L.rocJpegStreamParse.argtypes = [vp, C.c_size_t, vp]
    L.rocJpegStreamDestroy.argtypes = [vp]
    L.rocJpegCreate.argtypes = [i32, i32, C.POINTER(vp)]
    L.rocJpegDestroy.argtypes = [vp]
    L.rocJpegGetImageInfo.argtypes = [vp, vp, C.POINTER(C.c_uint8), C.POINTER(i32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
    L.rocJpegDecode.argtypes = [vp, vp, C.POINTER(RocJpegDecodeParams), C.POINTER(RocJpegImage)]
    L.rocJpegDecodeBatched.argtypes = [vp, C.POINTER(vp), i32, C.POINTER(RocJpegDecodeParams), C.POINTER(RocJpegImage)]
    L.rocJpegGetErrorName.argtypes = [i32]
    L.rocJpegGetErrorName.restype = C.c_char_p
    L.rocJpegB200SetProfiling.argtypes = [vp, i32]
    L.rocJpegB200GetStats.argtypes = [vp, C.POINTER(Stats)]
    L.rocJpegB200Prepare.argtypes = [vp, C.POINTER(vp), i32, C.POINTER(RocJpegDecodeParams), C.POINTER(RocJpegImage)]
    L.rocJpegB200Run.argtypes = [vp]
    L.rocJpegB200GetScaledImageInfo.argtypes = [vp, vp, i32, C.POINTER(C.c_uint8), C.POINTER(i32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
    L.rocJpegB200DecodeBatchedScaled.argtypes = [vp, C.POINTER(vp), i32, C.POINTER(RocJpegDecodeParams), C.POINTER(C.c_int32), C.POINTER(RocJpegImage)]
    L.rocJpegB200PrepareScaled.argtypes = [vp, C.POINTER(vp), i32, C.POINTER(RocJpegDecodeParams), C.POINTER(C.c_int32), C.POINTER(RocJpegImage)]
    L.rocJpegB200GetCoefficients.argtypes = [vp, i32, vp, C.c_size_t]
    L.rocJpegB200GetPlanes.argtypes = [vp, i32, vp, C.c_size_t]
    L.rocJpegB200StreamGetInfo.argtypes = [vp, C.POINTER(StreamInfo)]
    L.rocJpegB200StreamLoadFiles.argtypes = [C.POINTER(vp), C.POINTER(C.c_char_p), i32, i32, C.POINTER(i32)]
    L.rocJpegB200GetImageStatus.argtypes = [vp, i32, C.POINTER(C.c_uint32)]
    L.rocJpegB200GetScanStatus.argtypes = [vp, i32, C.POINTER(ScanStatus)]
    L.rocJpegB200GetDeviceSegment.argtypes = [vp, i32, C.c_uint32, vp, C.c_size_t, C.POINTER(C.c_uint32)]
    L.rocJpegB200ParseAndDecodeBatched.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(C.c_size_t), i32, C.POINTER(RocJpegDecodeParams),
                                                   C.POINTER(RocJpegImage), C.POINTER(C.c_double)]
    L.rocJpegB200StreamHostScan.argtypes = [vp, C.POINTER(HostScanInfo)]
    L.rocJpegB200StreamGetSegment.argtypes = [vp, C.c_uint32, vp, C.c_size_t, C.POINTER(C.c_uint32)]
    L.rocJpegB200StreamGetLastError.argtypes = [vp, C.c_char_p, C.c_size_t]
    L.rocJpegB200StreamGetQuantTable.argtypes = [vp, i32, vp]
    L.rocJpegB200StreamGetHuffmanTable.argtypes = [vp, i32, i32, vp, vp, C.POINTER(C.c_uint32)]
    L.rocJpegB200PlanShards.argtypes = [vp, i32, i32, vp]
    L.rocJpegB200PlanShardsPinned.argtypes = [vp, vp, i32, i32, vp]
    L.rocJpegB200GetDeviceCount.argtypes = [vp, C.POINTER(i32)]
    L.rocJpegB200Version.restype = C.c_char_p
    for name in EXPORTS + EXT_EXPORTS:
        if name not in ("rocJpegGetErrorName", "rocJpegB200Version"):
            getattr(L, name).restype = i32
    _lib = L
    return L


def plan_shards(costs, num_devices: int):
    """The longest-processing-time assignment rocJpegDecodeBatched uses when ROCJPEG_B200_DEVICES > 1."""
    import numpy as np

    c = np.ascontiguousarray(costs, dtype=np.uint64)
    out = np.zeros(len(c), dtype=np.int32)
    _check(load_library().rocJpegB200PlanShards(c.ctypes.data, len(c), num_devices, out.ctypes.data), "rocJpegB200PlanShards")
    return out


def plan_shards_pinned(costs, fixed, num_devices: int):
    """plan_shards with some images pinned to a device (fixed[i] >= 0): what the library does with destination buffers
    that already live on a peer device."""
    import numpy as np

    c = np.ascontiguousarray(costs, dtype=np.uint64)
    f = np.ascontiguousarray(fixed, dtype=np.int32)
    out = np.zeros(len(c), dtype=np.int32)
    _check(load_library().rocJpegB200PlanShardsPinned(c.ctypes.data, f.ctypes.data, len(c), num_devices, out.ctypes.data), "rocJpegB200PlanShardsPinned")
    return out


def load_files(streams, paths, io_threads: int = 0):
    """rocJpegB200StreamLoadFiles: read + parse paths[i] into streams[i] with I/O threads. Returns (status, per-file statuses)."""
    n = len(streams)
    hs = (C.c_void_p * n)(*[s.handle for s in streams])
    ps = (C.c_char_p * n)(*[os.fsencode(p) for p in paths])
    per = (C.c_int * n)()
    st = load_library().rocJpegB200StreamLoadFiles(hs, ps, n, io_threads, per)
    return st, list(per)


def error_name(status: int) -> str:
    return load_library().rocJpegGetErrorName(status).decode()


def _check(status: int, where: str):
    if status != SUCCESS:
        raise RocJpegError(status, where)


class JpegStream:
    """rocJpegStreamCreate / rocJpegStreamParse / rocJpegStreamDestroy."""

    def __init__(self):
        self.lib = load_library()
        self.handle = C.c_void_p()
        _check(self.lib.rocJpegStreamCreate(C.byref(self.handle)), "rocJpegStreamCreate")
        self._data = None

    def parse(self, data: bytes) -> int:
        """Returns the RocJpegStatus (0 on success); keeps `data` alive like the reference requires."""
        self._data = data
        return self.lib.rocJpegStreamParse(data, len(data), self.handle)

    def parse_ptr(self, address: int, length: int, keepalive=None) -> int:
        """rocJpegStreamParse on a raw host address (e.g. a slice of a page-locked arena)."""
        self._data = keepalive
        return self.lib.rocJpegStreamParse(C.c_void_p(address), length, self.handle)

    def info(self) -> StreamInfo:
        s = StreamInfo()
        _check(self.lib.rocJpegB200StreamGetInfo(self.handle, C.byref(s)), "rocJpegB200StreamGetInfo")
        return s

    def host_scan(self) -> HostScanInfo:
        """Host restatement of the GPU destuffing pass (tests only; needs the parsed bytes still alive)."""
        s = HostScanInfo()
        _check(self.lib.rocJpegB200StreamHostScan(self.handle, C.byref(s)), "rocJpegB200StreamHostScan")
        return s

    def segment(self, k: int) -> bytes:
        n = C.c_uint32()
        _check(self.lib.rocJpegB200StreamGetSegment(self.handle, k, None, 0, C.byref(n)), "segment size")
        buf = C.create_string_buffer(max(n.value, 1))
        _check(self.lib.rocJpegB200StreamGetSegment(self.handle, k, buf, n.value, C.byref(n)), "segment")
        return buf.raw[:n.value]

    def last_error(self) -> str:
        buf = C.create_string_buffer(512)
        _check(self.lib.rocJpegB200StreamGetLastError(self.handle, buf, len(buf)), "last error")
        return buf.value.decode("utf-8", "replace")

    def quant_table(self, tid: int):
        import numpy as np

        out = np.zeros(64, dtype=np.uint16)
        _check(self.lib.rocJpegB200StreamGetQuantTable(self.handle, tid, out.ctypes.data), "quant table")
        return out

    def huffman_table(self, is_ac: int, tid: int):
        bits = (C.c_uint8 * 16)()
        vals = (C.c_uint8 * 256)()
        n = C.c_uint32()
        _check(self.lib.rocJpegB200StreamGetHuffmanTable(self.handle, is_ac, tid, bits, vals, C.byref(n)), "huffman table")
        return bytes(bits), bytes(vals)[:n.value]

    def close(self):
        if self.handle:
            self.lib.rocJpegStreamDestroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def make_params(fmt, crop=(0, 0, 0, 0)) -> RocJpegDecodeParams:
    p = RocJpegDecodeParams()
    p.output_format = FMT[fmt] if isinstance(fmt, str) else int(fmt)
    p.crop_rectangle.left, p.crop_rectangle.top, p.crop_rectangle.right, p.crop_rectangle.bottom = crop
    return p


def output_channel_shapes(css: str, fmt: str, width: int, height: int):
    """(rows, valid bytes per row) per channel — samples/rocjpeg_samples_utils.h:318-399."""
    W, H = width, height
    if fmt == "rgb":
        return [(H, 3 * W)]
    if fmt == "rgb_planar":
        return [(H, W)] * 3
    if fmt == "y" or css == "400":
        return [(H, W)]
    if fmt == "native":
        return {"444": [(H, W)] * 3, "440": [(H, W), (H >> 1, W), (H >> 1, W)], "422": [(H, 2 * W)],
                "420": [(H, W), (H >> 1, W)], "411": [(H, W), (H, W >> 2), (H, W >> 2)]}[css]
    if fmt == "yuv_planar":
        return {"444": [(H, W)] * 3, "440": [(H, W), (H >> 1, W), (H >> 1, W)],
                "422": [(H, W), (H, W >> 1), (H, W >> 1)], "420": [(H, W), (H >> 1, W >> 1), (H >> 1, W >> 1)],
                "411": [(H, W), (H, W >> 2), (H, W >> 2)]}[css]
    raise ValueError((css, fmt))


class Decoder:
    """rocJpegCreate / rocJpegGetImageInfo / rocJpegDecode / rocJpegDecodeBatched / rocJpegDestroy."""

    def __init__(self, backend: int = BACKEND_HARDWARE, device_id: int = 0):
        self.lib = load_library()
        self.handle = C.c_void_p()
        st = self.lib.rocJpegCreate(backend, device_id, C.byref(self.handle))
        if st != SUCCESS:
            if self.handle:
                self.lib.rocJpegDestroy(self.handle)
                self.handle = C.c_void_p()
            raise RocJpegError(st, "rocJpegCreate")

    def image_info(self, stream: JpegStream):
        n = C.c_uint8()
        css = C.c_int()
        w = (C.c_uint32 * 4)()
        h = (C.c_uint32 * 4)()
        _check(self.lib.rocJpegGetImageInfo(self.handle, stream.handle, C.byref(n), C.byref(css), w, h), "rocJpegGetImageInfo")
        return n.value, css.value, list(w), list(h)

    def scaled_image_info(self, stream: JpegStream, scale_denom: int):
        """rocJpegB200GetScaledImageInfo: (num_components, subsampling, widths, heights) of a decode at 1/scale_denom."""
        n = C.c_uint8()
        css = C.c_int()
        w = (C.c_uint32 * 4)()
        h = (C.c_uint32 * 4)()
        _check(self.lib.rocJpegB200GetScaledImageInfo(self.handle, stream.handle, scale_denom, C.byref(n), C.byref(css), w, h),
               "rocJpegB200GetScaledImageInfo")
        return n.value, css.value, list(w), list(h)

    @staticmethod
    def _scales(scales, n):
        """int32 array of denominators (a ready ctypes array passes through), or None (all 1)."""
        if scales is None or isinstance(scales, C.Array):
            return scales
        if len(scales) != n:
            raise ValueError(f"{len(scales)} scale denominators for {n} pictures")
        return (C.c_int32 * n)(*[int(d) for d in scales])

    @staticmethod
    def _images(dests):
        arr = (RocJpegImage * len(dests))()
        for i, d in enumerate(dests):
            for c, (ptr, pitch) in enumerate(d):
                arr[i].channel[c] = ptr
                arr[i].pitch[c] = pitch
        return arr

    def decode(self, stream: JpegStream, params: RocJpegDecodeParams, dest) -> int:
        """dest: list of (device pointer, pitch) per channel. Returns RocJpegStatus."""
        img = self._images([dest])
        return self.lib.rocJpegDecode(self.handle, stream.handle, C.byref(params), img)

    def make_batch(self, streams, dests):
        """Pre-built argument arrays for decode_batched (what a C caller already holds), so a
        timed region around the call measures the library, not ctypes marshalling."""
        hs = (C.c_void_p * len(streams))(*[s.handle for s in streams])
        return (hs, self._images(dests), len(streams), list(streams))

    def decode_batched(self, streams, params: RocJpegDecodeParams, dests=None) -> int:
        hs, imgs, n, _ = streams if dests is None else self.make_batch(streams, dests)
        return self.lib.rocJpegDecodeBatched(self.handle, hs, n, C.byref(params), imgs)

    def decode_batched_scaled(self, streams, params: RocJpegDecodeParams, dests, scales) -> int:
        """rocJpegB200DecodeBatchedScaled: picture i decoded at 1/scales[i] (scales None: all full size). dests and the crop
        rectangle are in scaled units (scaled_image_info). Returns RocJpegStatus."""
        hs, imgs, n, _ = streams if dests is None else self.make_batch(streams, dests)
        return self.lib.rocJpegB200DecodeBatchedScaled(self.handle, hs, n, C.byref(params), self._scales(scales, n), imgs)

    def make_sources(self, addresses, lengths):
        """Argument arrays (data pointers, lengths) for parse_and_decode_batched."""
        n = len(addresses)
        return ((C.c_void_p * n)(*addresses), (C.c_size_t * n)(*lengths))

    def parse_and_decode_batched(self, batch, sources, params: RocJpegDecodeParams):
        """rocJpegStreamParse per image + one rocJpegDecodeBatched, looped in C (the caller's loop of the reference's
        batched sample). Returns (status, seconds spent in the parse loop)."""
        hs, imgs, n, _ = batch
        ptrs, lens = sources
        sec = C.c_double()
        st = self.lib.rocJpegB200ParseAndDecodeBatched(self.handle, hs, ptrs, lens, n, C.byref(params), imgs, C.byref(sec))
        return st, sec.value

    # ---- extension taps -------------------------------------------------
    def prepare(self, streams, params, dests, scales=None) -> int:
        """rocJpegB200Prepare, or rocJpegB200PrepareScaled when `scales` (one denominator per picture) is given."""
        hs = (C.c_void_p * len(streams))(*[s.handle for s in streams])
        imgs = self._images(dests)
        if scales is None:
            return self.lib.rocJpegB200Prepare(self.handle, hs, len(streams), C.byref(params), imgs)
        return self.lib.rocJpegB200PrepareScaled(self.handle, hs, len(streams), C.byref(params), self._scales(scales, len(streams)), imgs)

    def run(self) -> int:
        return self.lib.rocJpegB200Run(self.handle)

    def num_devices(self) -> int:
        n = C.c_int()
        _check(self.lib.rocJpegB200GetDeviceCount(self.handle, C.byref(n)), "rocJpegB200GetDeviceCount")
        return n.value

    def set_profiling(self, level):
        """0/False off, 1/True per-stage events, 2 first/last event only (total_ms)."""
        self.lib.rocJpegB200SetProfiling(self.handle, int(level))

    def stats(self) -> Stats:
        s = Stats()
        _check(self.lib.rocJpegB200GetStats(self.handle, C.byref(s)), "rocJpegB200GetStats")
        return s

    def coefficients(self, index: int, count: int):
        import numpy as np

        out = np.zeros(count, dtype=np.int16)
        _check(self.lib.rocJpegB200GetCoefficients(self.handle, index, out.ctypes.data, count), "rocJpegB200GetCoefficients")
        return out

    def scan_status(self, index: int) -> ScanStatus:
        s = ScanStatus()
        _check(self.lib.rocJpegB200GetScanStatus(self.handle, index, C.byref(s)), "rocJpegB200GetScanStatus")
        return s

    def image_status(self, index: int) -> int:
        """SCAN_* | DECODE_* flags of image `index` of the last decode call."""
        f = C.c_uint32()
        _check(self.lib.rocJpegB200GetImageStatus(self.handle, index, C.byref(f)), "rocJpegB200GetImageStatus")
        return f.value

    def device_segment(self, index: int, k: int) -> bytes:
        """Restart interval k of image `index` as the GPU destuffing pass left it in device memory."""
        n = C.c_uint32()
        _check(self.lib.rocJpegB200GetDeviceSegment(self.handle, index, k, None, 0, C.byref(n)), "device segment size")
        buf = C.create_string_buffer(max(n.value, 1))
        _check(self.lib.rocJpegB200GetDeviceSegment(self.handle, index, k, buf, n.value, C.byref(n)), "device segment")
        return buf.raw[:n.value]

    def planes(self, index: int, count: int):
        import numpy as np

        out = np.zeros(count, dtype=np.uint8)
        _check(self.lib.rocJpegB200GetPlanes(self.handle, index, out.ctypes.data, count), "rocJpegB200GetPlanes")
        return out

    def close(self):
        if self.handle:
            self.lib.rocJpegDestroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

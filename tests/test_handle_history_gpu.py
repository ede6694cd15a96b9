"""Call history (-m gpu): what a decode writes must depend on its own inputs only - not on what its handle, or another handle,
did before. Device memory is reused across calls by design (grow-only arenas that are never cleared, counter sets one call
leaves zeroed for the next, crops that leave parts of the plane arena unwritten), so every call of a menu - whole pictures,
crops, reduced-size and resized decodes, failing calls, entropy-stage schedules, lane counts, Prepare / Run - is run on
poisoned handles (ROCJPEG_B200_POISON: new arenas and staging start as a chosen byte, not as cudaMalloc's zeros), after decoys
that leave wrong values exactly where a crop must not read, in shuffled sequences, after failures and from several threads
at once, and must give the same destination bytes, status and per-picture flags every time. Expected values come from the
oracle, the JFIF restatement, the reduced-size oracle and Pillow, computed once per module."""
import contextlib
import functools
import io
import json
import os
import random
import threading
from dataclasses import dataclass, field

import numpy as np
import pytest
from PIL import Image

from rocjpeg_b200 import api, datagen

import gpu_util as gu
import jfif_oracle as jo
import scaled_oracle as so
from test_resize_gpu import expected_decode, pillow_resize

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden")
with open(os.path.join(GOLDEN, "golden.json")) as _f:
    CASES = sorted(json.load(_f)["cases"])
REF, LJ = api.COLOR_REFERENCE, api.COLOR_LIBJPEG


def load(name):
    with open(os.path.join(GOLDEN, name + ".jpg"), "rb") as f:
        return f.read()


@dataclass(frozen=True)
class Recipe:
    """How a generated picture was made: a decoy is the same geometry, subsampling and restart layout with other pixels."""
    w: int
    h: int
    css: str
    seed: int
    restart_rows: int = 0

    @functools.lru_cache(maxsize=None)
    def data(self):
        return datagen.make_jpeg(self.w, self.h, self.css, seed=self.seed, restart_rows=self.restart_rows)

    @functools.lru_cache(maxsize=None)
    def decoys(self):
        flat = np.empty((self.h, self.w, 3), np.uint8)
        flat[...] = (201, 37, 96)
        return [datagen.make_jpeg(self.w, self.h, self.css, seed=self.seed + 5000, restart_rows=self.restart_rows),
                datagen.encode_jpeg(flat, self.css, restart_rows=self.restart_rows)]


@dataclass
class Entry:
    """One call of the menu and what it must produce."""
    name: str
    datas: list
    fmt: str
    conv: int = REF
    crop: tuple = (0, 0, 0, 0)
    scales: list = None
    resize: tuple = None          # (sizes, filters)
    prepare: bool = False         # Prepare, then two Runs
    env: dict = field(default_factory=dict)
    recipes: list = None          # the pictures' recipes (crop, scaled and resized-crop entries: decoys)
    pad: int = 0
    mis: int = 0
    status: int = api.SUCCESS
    want: list = None             # per picture: whole channel arrays (rows, pitch), FILL outside what the call writes
    flags: list = None            # per picture: rocJpegB200GetImageStatus
    truncated: int = 0
    fallback: bool = False        # the entropy stage must have run more than one synchronisation round
    from_fresh_handle: bool = False   # a truncated picture: expected bytes are those of the same call on a fresh handle

    @property
    def partial(self):
        return self.recipes is not None

    @property
    def big(self):
        return len(self.datas) >= 8 or any(len(d) > 400_000 for d in self.datas)


def layout(orc, e, datas=None, crop=None):
    """Per picture: (shapes, pitches) of its destination channels."""
    datas = e.datas if datas is None else datas
    crop = e.crop if crop is None else crop
    out = []
    for k, data in enumerate(datas):
        if e.resize:
            W, H = e.resize[0][k]
            shapes = [(H, 3 * W)] if e.fmt == "rgb" else [(H, W)] * (3 if e.fmt == "rgb_planar" else 1)
            out.append((shapes, [shapes[0][1] + e.pad] * len(shapes)))
        else:
            rc, info = orc.parse(data)
            d = e.scales[k] if e.scales else 1
            # a call refused at validation: destinations of the whole picture, which it must leave untouched
            alloc_crop = (0, 0, 0, 0) if e.status == api.INVALID_PARAMETER else crop
            out.append(gu.output_layout(orc, so.scaled_info(info, d), e.fmt, alloc_crop, e.pad))
    return out


def expected(orc, jorc, sorc, e):
    """Whole destination arrays of every picture of a call that succeeds, from the oracles."""
    out = []
    for k, (data, (shapes, pitches)) in enumerate(zip(e.datas, layout(orc, e))):
        d = e.scales[k] if e.scales else 1
        if e.status == api.INVALID_PARAMETER:
            out.append([np.full((rows, p), gu.FILL, np.uint8) for (rows, _), p in zip(shapes, pitches)])
        elif e.resize:
            src = expected_decode(orc, jorc, sorc, e.conv, data, e.fmt, d)
            if e.crop != (0, 0, 0, 0):
                src = src[e.crop[1]:e.crop[3], e.crop[0]:e.crop[2]]
            size, filt = e.resize[0][k], e.resize[1][k]
            px = pillow_resize(src, size, filt)
            arrs = [np.full((rows, p), gu.FILL, np.uint8) for (rows, _), p in zip(shapes, pitches)]
            W, H = size
            if e.fmt == "rgb":
                arrs[0][:, :3 * W] = px.reshape(H, 3 * W)
            else:
                for c, a in enumerate(arrs):
                    a[:, :W] = px[:, :, c]
            out.append(arrs)
        elif e.conv == LJ and e.fmt in ("rgb", "rgb_planar"):
            out.append(jorc.decode(data, e.fmt, d, e.crop, pitches, fill=gu.FILL)[1])
        elif d == 1:
            out.append(orc.decode(data, e.fmt, e.crop, pitches=pitches, fill=gu.FILL)[1])
        else:
            out.append(sorc.decode_scaled(data, d, e.fmt, e.crop, pitches, fill=gu.FILL)[1])
    return out


@contextlib.contextmanager
def knobs(env):
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def stream(data):
    s = api.JpegStream()
    assert s.parse(data) == api.SUCCESS
    return s


class Call:
    """One entry (or a decoy of it) with its destinations. They are allocated here, before any call, and the callers
    synchronise before calling (test_stream_order_gpu.py tests the call's own ordering after torch's default stream)."""

    def __init__(self, orc, e, datas=None, crop=None):
        import torch

        self.e = e
        self.datas = e.datas if datas is None else datas
        self.crop = e.crop if crop is None else crop
        self.layout = layout(orc, e, self.datas, self.crop)
        self.bufs = [[torch.full((rows * p + e.mis + 64,), gu.FILL, dtype=torch.uint8, device="cuda") for (rows, _), p in zip(*lay)]
                     for lay in self.layout]

    def refill(self):
        for bufs in self.bufs:
            for b in bufs:
                b.fill_(gu.FILL)

    def start(self, dec):
        """Parse (from pageable bytes) and call; Prepare entries stop after Prepare. Returns the status."""
        e = self.e
        dec.set_color_convention(e.conv)
        self.streams = [stream(d) for d in self.datas]
        dests = [[(b.data_ptr() + e.mis, p) for b, p in zip(bufs, lay[1])] for bufs, lay in zip(self.bufs, self.layout)]
        params = api.make_params(e.fmt, self.crop)
        with knobs(e.env):
            if e.resize:
                sizes, filters = e.resize
                if e.prepare:
                    return dec.prepare_resized(self.streams, params, dests, sizes, filters, e.scales)
                return dec.decode_batched_resized(self.streams, params, dests, sizes, filters, e.scales)
            if e.prepare:
                return dec.prepare(self.streams, params, dests, e.scales)
            return dec.decode_batched_scaled(self.streams, params, dests, e.scales)

    def outcome(self, dec, st):
        """(status, per-picture flags or None, truncated pictures, sync rounds) of the call just made."""
        if st not in (api.SUCCESS, api.BAD_JPEG):
            return st, None, None, None
        s = dec.stats()
        return st, [dec.image_status(i) for i in range(len(self.datas))], s.truncated_images, s.sync_rounds

    def fetch(self):
        return [gu.fetch(bufs, lay[1], lay[0], self.e.mis) for bufs, lay in zip(self.bufs, self.layout)]

    def mismatches(self, outcome, what):
        """What differs from the entry's expected result, as a list of messages (empty: exact)."""
        e = self.e
        st, flags, truncated, rounds = outcome
        bad = []
        if st != e.status:
            return [f"{what}: status {api.STATUS.get(st, st)}, want {api.STATUS.get(e.status, e.status)}"]
        if flags is not None and (flags != e.flags or truncated != e.truncated):
            bad.append(f"{what}: image status {flags} truncated {truncated}, want {e.flags} truncated {e.truncated}")
        if e.fallback and rounds is not None and rounds <= 1:
            bad.append(f"{what}: {rounds} sync round(s): the entropy-stage fallback was not exercised")
        try:
            got = self.fetch()
        except AssertionError as x:
            return bad + [f"{what}: {x}"]
        for k, (g, w) in enumerate(zip(got, e.want)):
            try:
                gu.assert_same(g, w, f"{what} picture {k}")
            except AssertionError as x:
                bad.append(str(x))
        return bad


def run_entry(orc, dec, e, what):
    """Run one entry on `dec` (Prepare entries: Prepare and two Runs, destinations refilled in between) and check every
    outcome; returns the mismatches."""
    import torch

    c = Call(orc, e)
    torch.cuda.synchronize()
    st = c.start(dec)
    if not e.prepare:
        return c.mismatches(c.outcome(dec, st), what)
    assert st == api.SUCCESS, (what, st)
    bad = []
    for rep in range(2):
        if rep:
            c.refill()
            torch.cuda.synchronize()
        with knobs(e.env):
            st = dec.run()
        bad += c.mismatches(c.outcome(dec, st), f"{what} run {rep}")
    return bad


def run_decoy(orc, dec, e):
    """Decode pictures of the entry's layout with other pixels, in the entry's own format, scales and resize, cropped to
    the whole picture minus one row: the plane arena then holds wrong values wherever the entry's own call leaves it
    unwritten (a whole-picture call would take the fused or direct paths and leave the arena alone)."""
    import torch

    for k in range(2):
        datas = [r.decoys()[k] for r in e.recipes]
        d = e.scales[0] if e.scales else 1
        w, h = -(-e.recipes[0].w // d), -(-e.recipes[0].h // d)
        c = Call(orc, Entry(e.name + " decoy", datas, e.fmt, e.conv, scales=e.scales, resize=e.resize, env=e.env), datas, (0, 0, w, h - 1))
        torch.cuda.synchronize()
        st = c.start(dec)
        assert st == api.SUCCESS, (e.name, "decoy", st)


# ---------------------------------------------------------------------------------------------------------------- menu

def truncated_batch():
    """test_truncated_picture_resized_from_its_decode's pair: a clean 4:4:4 picture and a 4:2:0 one cut 37 bytes into its
    ninth restart interval."""
    whole = datagen.make_jpeg(320, 240, "420", seed=5, restart_rows=1)
    i0 = stream(whole).info()
    scan = whole[i0.scan_offset:]
    marks = [k for k in range(len(scan) - 1) if scan[k] == 0xFF and 0xD0 <= scan[k + 1] <= 0xD7]
    return [load("synth_444_500x375"), whole[:i0.scan_offset + marks[8] + 2 + 37]]


def optimised(seed):
    """A small picture with optimised Huffman tables (libjpeg's two-pass table choice): every seed its own table set."""
    rng = np.random.default_rng(seed)
    w, h = int(rng.integers(40, 200)), int(rng.integers(30, 160))
    bio = io.BytesIO()
    Image.fromarray(datagen.synth_image(w, h, seed)).save(bio, format="JPEG", quality=int(rng.integers(50, 98)), optimize=True,
                                                         subsampling=int(seed % 3))
    return bio.getvalue()


def boundary_crops(bx, by):
    """Edges on chroma-block boundaries (bx, by luma samples per chroma block) and one sample either side."""
    return [(2 * bx, 2 * by, 6 * bx, 5 * by), (2 * bx - 1, 2 * by - 1, 6 * bx + 1, 5 * by + 1), (2 * bx + 1, 2 * by + 1, 6 * bx - 1, 5 * by - 1)]


def build_menu():
    M = []
    golden = [load(n) for n in CASES]
    # whole pictures
    for fmt in ("native", "yuv_planar", "y", "rgb", "rgb_planar"):
        M.append(Entry(f"golden {fmt}", golden, fmt, pad=3 if fmt == "rgb" else 0, mis=1 if fmt == "yuv_planar" else 0))
    for fmt in ("rgb", "rgb_planar"):
        M.append(Entry(f"golden {fmt} libjpeg", golden, fmt, LJ, pad=5 if fmt == "rgb_planar" else 0))
    # crops: edges on chroma-block boundaries (16 luma samples is one for every subsampling) and one sample either side
    rec = [Recipe(200, 150, css, 30 + i) for i, css in enumerate(("420", "422", "440", "444"))]
    for crop in boundary_crops(16, 16):
        for conv, fmt in ((LJ, "rgb"), (LJ, "rgb_planar"), (REF, "rgb"), (REF, "yuv_planar"), (REF, "native")):
            M.append(Entry(f"boundary crop {crop} {fmt} conv={conv}", [r.data() for r in rec], fmt, conv, crop, recipes=rec, pad=3))
    # ... on a picture wide enough for chroma blocks in three IDCT tiles of 32 blocks: the edges on the tile boundaries
    for css in ("420", "422"):
        r = Recipe(1072, 96, css, 40)
        for conv in (LJ, REF):
            M.append(Entry(f"tile-boundary crop {css} conv={conv}", [r.data()], "rgb", conv, (512, 16, 1024, 80), recipes=[r]))
    # restart intervals outside the crop are not entropy-decoded
    for css, mcu in (("420", 16), ("440", 16), ("422", 8)):
        r = Recipe(300, 200, css, 11, restart_rows=1)
        for crop in ((0, 3 * mcu, 300, 5 * mcu), (17, 3 * mcu + 1, 201, 5 * mcu - 1)):
            for conv in (LJ, REF):
                M.append(Entry(f"dri crop {css} {crop} conv={conv}", [r.data()], "rgb", conv, crop, recipes=[r]))
    # reduced-size crops (crop in scaled units; a chroma block is 16/d output samples of 4:2:0)
    rec = [Recipe(500, 375, "420", 50, restart_rows=2), Recipe(500, 375, "422", 51), Recipe(500, 375, "444", 52)]
    for d in (2, 4, 8):
        B = 16 // d
        for crop in ((3 * B, 2 * B, 11 * B, 9 * B), (3 * B + 1, 2 * B - 1, 11 * B - 1, 9 * B + 1)):
            for conv in (LJ, REF):
                M.append(Entry(f"scaled crop 1/{d} {crop} conv={conv}", [r.data() for r in rec], "rgb", conv, crop, [d] * 3, recipes=rec))
    # mixed scales, resized batches with crop and scale
    scales = [(1, 2, 4, 8)[i % 4] for i in range(len(golden))]
    M.append(Entry("golden mixed scales rgb", golden, "rgb", REF, scales=scales, pad=2))
    M.append(Entry("golden mixed scales rgb_planar libjpeg", golden, "rgb_planar", LJ, scales=scales))
    M.append(Entry("golden mixed scales yuv_planar", golden, "yuv_planar", REF, scales=scales, mis=3))
    sizes = [((37 * i) % 150 + 1, (53 * i) % 120 + 1) for i in range(len(golden))]
    M.append(Entry("golden resized", golden, "rgb", REF, scales=scales, resize=(sizes, [api.FILTERS[i % 5] for i in range(len(golden))])))
    for d, crop in ((1, (16, 32, 400, 300)), (2, (8, 16, 200, 150)), (4, (3, 5, 101, 77))):
        cw, ch = crop[2] - crop[0], crop[3] - crop[1]
        rsz = ([(cw * 2 // 3, ch * 3 // 5), (cw + 5, ch * 2 + 1), (224, 224)], [api.FILTER_LANCZOS, api.FILTER_BICUBIC, api.FILTER_HAMMING])
        for conv, fmt in ((LJ, "rgb"), (REF, "rgb_planar"), (REF, "y")):
            M.append(Entry(f"resized crop 1/{d} {crop} {fmt} conv={conv}", [r.data() for r in rec], fmt, conv, crop, [d] * 3, rsz, recipes=rec, pad=1))
    # arena growth: a 3840x2160 4:2:0 picture
    big = datagen.make_jpeg(3840, 2160, "420", seed=21)
    M.append(Entry("4k rgb", [big], "rgb"))
    M.append(Entry("4k rgb libjpeg", [big], "rgb", LJ))
    M.append(Entry("4k yuv_planar", [big], "yuv_planar"))
    r = Recipe(3840, 2160, "420", 21)
    M.append(Entry("4k crop libjpeg", [big], "rgb_planar", LJ, (1001, 777, 2999, 1601), recipes=[r]))
    # pictures with optimised Huffman tables: 24 table sets, more than the parser's process-wide cache of 16 holds
    opt = [optimised(900 + k) for k in range(24)]
    for k, (conv, fmt) in enumerate(((REF, "rgb"), (REF, "yuv_planar"), (LJ, "rgb"), (REF, "native"), (REF, "y"), (LJ, "rgb_planar"))):
        M.append(Entry(f"optimised tables {k} {fmt} conv={conv}", opt[4 * k:4 * k + 4], fmt, conv))
    # failing calls
    trunc = truncated_batch()
    M.append(Entry("truncated", trunc, "rgb", status=api.BAD_JPEG, from_fresh_handle=True))
    M.append(Entry("truncated resized", trunc, "rgb", resize=([(200, 150), (224, 224)], [api.FILTER_BICUBIC, api.FILTER_LANCZOS]),
                   status=api.BAD_JPEG, from_fresh_handle=True))
    M.append(Entry("crop outside the picture", [load("synth_422_123x77"), load("synth_420_64x64")], "rgb", crop=(40, 0, 70, 20),
                   status=api.INVALID_PARAMETER))
    M.append(Entry("resized crop outside the picture", [load("synth_444_123x77")], "rgb_planar", LJ, (100, 50, 130, 60),
                   resize=([(32, 32)], [api.FILTER_BILINEAR]), status=api.INVALID_PARAMETER))
    # entropy-stage schedules
    fb = [datagen.make_jpeg(500, 375, css, seed=700 + i) for i, css in enumerate(("444", "422", "420", "444"))]
    M.append(Entry("fallback (halo 1)", fb, "rgb_planar", env={"ROCJPEG_B200_HALO": "1", "ROCJPEG_B200_SUBSEQ": "32"}, fallback=True))
    M.append(Entry("one sync round", [load("synth_444_500x375")], "rgb", env={"ROCJPEG_B200_SYNC_ROUNDS": "1", "ROCJPEG_B200_SUBSEQ": "32"}))
    M.append(Entry("separate entropy kernels", fb, "yuv_planar", env={"ROCJPEG_B200_NO_K1_FUSE": "1"}))
    M.append(Entry("separate tile scan", golden, "rgb", LJ, env={"ROCJPEG_B200_NO_INLINE_SCAN": "1"}))
    M.append(Entry("tiled DC kernels", golden, "native", env={"ROCJPEG_B200_NO_K1_DC": "1"}))
    # lanes (lanes 4-7 are created without preallocation: they grow on demand)
    for lanes in ("1", "4", "8"):
        M.append(Entry(f"{lanes} lanes", golden, "rgb_planar", env={"ROCJPEG_B200_LANES": lanes}))
    # Prepare, then two Runs
    M.append(Entry("prepare", golden, "rgb", LJ, scales=scales, prepare=True))
    M.append(Entry("prepare resized", [r.data() for r in rec], "rgb", REF, (8, 16, 200, 150), [2] * 3,
                   ([(100, 80), (61, 97), (224, 224)], [api.FILTER_BOX, api.FILTER_BILINEAR, api.FILTER_LANCZOS]), prepare=True))
    return M


@pytest.fixture(scope="module")
def menu(orc):
    """The menu with every entry's expected result (oracles on the main thread; a truncated picture's bytes from the same
    call on a fresh handle, whose rows before the cut must equal the oracle's)."""
    import torch

    assert torch.cuda.is_available()
    torch.cuda.set_device(0)
    jorc, sorc = jo.JfifOracle(orc), so.ScaledOracle(orc)
    M = build_menu()
    fresh = api.Decoder(api.BACKEND_HARDWARE, 0)
    try:
        for e in M:
            e.flags = [0] * len(e.datas)
            if not e.from_fresh_handle:
                e.want = expected(orc, jorc, sorc, e)
                continue
            c = Call(orc, e)
            torch.cuda.synchronize()
            st, flags, truncated, _ = c.outcome(fresh, c.start(fresh))
            assert st == e.status and flags[1] & api.DECODE_SHORT and truncated == 1, (e.name, st, flags, truncated)
            e.flags, e.truncated, e.want = flags, truncated, c.fetch()
            good = Entry(e.name, e.datas[:1], e.fmt, resize=e.resize and ([e.resize[0][0]], [e.resize[1][0]]))
            gu.assert_same(e.want[0], expected(orc, jorc, sorc, good)[0], f"{e.name}: the clean picture")
            if not e.resize:   # the restart intervals before the cut (8 MCU rows of 16), less one MCU row for the chroma filter
                rc, info = orc.parse(e.datas[1])
                head = orc.decode(e.datas[1], "rgb", fill=gu.FILL)[1][0][:112]
                assert np.array_equal(e.want[1][0][:112, :3 * info.width], head[:, :3 * info.width]), f"{e.name}: rows before the cut"
    finally:
        fresh.close()
    return M


@pytest.fixture
def poisoned(monkeypatch):
    """Handles created from here on start with empty arenas (growing call by call) filled with the poison byte."""
    def new(byte=0x5A):
        monkeypatch.setenv("ROCJPEG_B200_POISON", hex(byte))
        monkeypatch.setenv("ROCJPEG_B200_PREALLOC_MB", "0")
        return api.Decoder(api.BACKEND_HARDWARE, 0)
    return new


# --------------------------------------------------------------------------------------------------------------- tests

@pytest.mark.parametrize("byte", [0x5A, 0xFF])
def test_poisoned_fresh_handle(orc, menu, poisoned, byte):
    """Every entry once, each on a new handle whose arenas start as the poison byte (0xFF: the scan's marker byte and the
    block records' "never decoded" fill)."""
    bad = []
    for e in menu:
        dec = poisoned(byte)
        try:
            bad += run_entry(orc, dec, e, f"{e.name} poison={byte:#x}")
        finally:
            dec.close()
    assert not bad, "\n".join(bad)


def test_decoy_before_every_partial_call(orc, menu, poisoned):
    """test_jfif_gpu.check_crops decodes the whole picture before each crop, so the blocks a crop wrongly skips still hold
    the right values. Here they hold a decoy's: the same layout with other pixels (another seed, then a flat picture)."""
    dec = poisoned()
    bad = []
    try:
        for e in menu:
            if not e.partial:
                continue
            run_decoy(orc, dec, e)
            bad += run_entry(orc, dec, e, f"{e.name} after decoys")
    finally:
        dec.close()
    assert not bad, "\n".join(bad)


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_seeded_call_sequences(orc, menu, poisoned, seed):
    """The whole menu shuffled on one handle, large and small batches alternating: arenas grow, and are reused with larger
    stale contents than the next call writes."""
    order = list(menu)
    random.Random(seed).shuffle(order)
    big, small = [e for e in order if e.big], [e for e in order if not e.big]
    seq = []
    while big or small:
        seq += [x.pop() for x in (big, small) if x]
    dec = poisoned()
    bad = []
    try:
        for k, e in enumerate(seq):
            bad += run_entry(orc, dec, e, f"seed {seed} call {k} {e.name}")
    finally:
        dec.close()
    assert not bad, "\n".join(bad)


def test_failure_then_success(orc, menu, poisoned):
    import torch

    by = {e.name: e for e in menu}
    good_crop, good_whole = by[f"boundary crop {boundary_crops(16, 16)[0]} rgb conv={LJ}"], by["golden rgb"]
    dec = poisoned()
    bad = []
    try:
        # refused at validation: nothing written, nothing left to Run, the next call exact
        bad += run_entry(orc, dec, by["crop outside the picture"], "validation failure")
        assert dec.run() == api.NOT_INITIALIZED
        bad += run_entry(orc, dec, good_crop, "after a validation failure")
        # a truncated batch still leaves a decoded batch behind: Run replays it, status, flags and bytes
        e = by["truncated"]
        c = Call(orc, e)
        torch.cuda.synchronize()
        bad += c.mismatches(c.outcome(dec, c.start(dec)), "truncated")
        c.refill()
        torch.cuda.synchronize()
        bad += c.mismatches(c.outcome(dec, dec.run()), "truncated, run again")
        bad += run_entry(orc, dec, good_crop, "after a truncated batch")
        # the entropy-stage fallback, then the fused path
        bad += run_entry(orc, dec, by["fallback (halo 1)"], "fallback")
        bad += run_entry(orc, dec, good_whole, "after the fallback")
        assert dec.stats().fused_blocks > 0
        # Prepare(A), Decode(B): Run replays B and leaves A's destinations alone
        a, b = by["prepare"], good_crop
        ca, cb = Call(orc, a), Call(orc, b)
        torch.cuda.synchronize()
        assert ca.start(dec) == api.SUCCESS
        bad += cb.mismatches(cb.outcome(dec, cb.start(dec)), "decode after prepare")
        cb.refill()
        torch.cuda.synchronize()
        bad += cb.mismatches(cb.outcome(dec, dec.run()), "run after prepare, decode")
        for k, bufs in enumerate(ca.bufs):
            for t in bufs:
                if not bool((t == gu.FILL).all()):
                    bad.append(f"run after prepare, decode: the prepared batch's picture {k} was written")
    finally:
        dec.close()
    assert not bad, "\n".join(bad)


@pytest.mark.parametrize("deferred", ["0", "1"])
def test_concurrent_handles(orc, menu, monkeypatch, deferred):
    """Four threads, one handle each, decode different seeded slices of the menu at the same time (ctypes releases the
    GIL): the page-locked staging pool and the Huffman table cache - which evicts tables other handles still use - are
    shared by all of them."""
    import torch

    monkeypatch.setenv("ROCJPEG_B200_POISON", "0x5A")
    monkeypatch.setenv("ROCJPEG_B200_PREALLOC_MB", "0")
    monkeypatch.setenv("ROCJPEG_B200_DEFERRED_COPY", deferred)
    eligible = [e for e in menu if not e.env and not e.prepare]   # environment knobs are process-wide
    assert len({stream(d).huffman_table(1, 0) for e in eligible for d in e.datas}) >= 20   # more table sets than the cache holds
    slices = []
    for t in range(4):
        order = list(eligible)
        random.Random(100 + t).shuffle(order)
        slices.append(order[:len(order) * 2 // 3])
    decs = [api.Decoder(api.BACKEND_HARDWARE, 0) for _ in range(4)]
    calls = [[Call(orc, e) for e in sl] for sl in slices]
    torch.cuda.synchronize()
    outcomes = [[] for _ in range(4)]
    errors = [None] * 4

    def work(t):
        try:
            for c in calls[t]:
                outcomes[t].append(c.outcome(decs[t], c.start(decs[t])))
        except Exception as x:   # reported after the join
            errors[t] = repr(x)

    threads = [threading.Thread(target=work, args=(t,)) for t in range(4)]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    bad = []
    try:
        for t in range(4):
            assert errors[t] is None, f"thread {t}: {errors[t]}"
            for k, (c, out) in enumerate(zip(calls[t], outcomes[t])):
                bad += c.mismatches(out, f"thread {t} call {k} {c.e.name}")
    finally:
        for d in decs:
            d.close()
    assert not bad, "\n".join(bad)

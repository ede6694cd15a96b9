"""Stream order (-m gpu): a call must not touch the caller's destinations before the work the caller has already enqueued
on the device's legacy default stream - torch's default stream - is done with them. The library's streams are
non-blocking, so each call orders them after that work itself. Every case queues a bounded spin (torch.cuda._sleep) and
then an operation on a destination on the legacy default stream, checks that the spin is still running, makes one library
call, synchronises and compares the whole buffers (canaries included) with the oracles:

- write after write: the queued operation fills the channels; the decode must land after it;
- write after read: the queued operation copies the destination out; the copy must see what was there before the call;
- the caching allocator's idiom: the queued operation reads a tensor that is then freed, and the destination is allocated
  into the freed block, as torch.empty does in a training loop; the reader must see the freed tensor's contents;
- read after return: the destination read on the default stream right after the call, without a synchronise.

Nothing may synchronise the device between the spin and the call, or the hazard would pass unseen. So each case runs
the same call once beforehand with nothing pending: arenas, lanes and staging already have their size, and the call under
test allocates nothing (a cudaFree synchronises the device), and neither does the test inside the window beyond
reusing a block the caching allocator holds. It also runs the queued operation once outside that window:
under CUDA's lazy module loading the first launch of a kernel loads its module, which can synchronise the context (the
byte fill of a view one byte off alignment is a kernel of its own). And garbage collection is off in the window: a
collection could destroy an earlier test's stream handles, whose page-locked staging cudaFreeHost releases. An event
recorded right behind the spin must still be pending when the call starts."""
import gc
import os
import re
from dataclasses import dataclass

import numpy as np
import pytest

from rocjpeg_b200 import api

import gpu_util as gu
import jfif_oracle as jo
import scaled_oracle as so
from test_handle_history_gpu import CASES, Entry, expected, knobs, layout, load, stream, truncated_batch

pytestmark = pytest.mark.gpu

SLEEP_CYCLES = 120_000_000   # the queued spin: about 60 ms at the B200's 1965 MHz SM clock, far longer than any call here
OVERWRITE = 0x3C             # what the queued fill writes (the canaries stay gu.FILL)
# The allocator idiom's block (channel + canaries): larger than the 20 MiB segments the caching allocator carves smaller
# blocks from, so the freed block is the only free one that fits and the next allocation of that size gets it.
ALLOC_BYTES = 32 << 20
REF, LJ = api.COLOR_REFERENCE, api.COLOR_LIBJPEG
HAZARDS = ["write_after_write", "write_after_read", "allocator", "read_after_return"]


@dataclass
class Case:
    """One library call. `entry` describes the pictures, format and destinations (test_handle_history_gpu's layout and
    oracles; pitch padding 0, so the call writes every byte of each channel); `watch` are the pictures the hazard is put
    on (the allocator idiom takes the last one's first channel)."""
    name: str
    entry: Entry
    call: str = "batched"        # "decode" (rocJpegDecode), "batched", "scaled", "resized", "prepare" (Prepare, then two Runs)
    watch: list = None           # None: every picture
    status: int = api.SUCCESS
    fused: bool = None           # True: the fused IDCT + colour kernel served the call
    lanes: int = None            # the lanes the call must have used
    sharded: bool = False        # ROCJPEG_B200_DEVICES=2
    devices: int = None          # the devices that must have decoded a share
    dst_device: int = 0          # where the destinations live, and the device whose default stream holds the pending work
    pageable_deferred: bool = False


def big_batch():
    return [load(n) for n in CASES]


def build_cases():
    whole_420 = load("synth_420_500x375_dri7")   # 3 x 500 bytes per RGB row: 4-byte aligned rows
    trio = [whole_420, load("synth_444_500x375"), load("synth_422_500x375")]
    C = [
        Case("decode rgb aligned (k23_warp)", Entry("", [whole_420], "rgb"), call="decode", fused=True),
        Case("decode rgb misaligned (k23_fused)", Entry("", [whole_420], "rgb", mis=1), call="decode", fused=True),
        Case("yuv_planar (IDCT direct stores)", Entry("", trio, "yuv_planar"), fused=False),
        Case("y (IDCT direct stores)", Entry("", trio, "y"), fused=False),
        Case("rgb crop (k3_output)", Entry("", trio, "rgb", crop=(17, 9, 301, 203)), fused=False),
        Case("native (k3_output)", Entry("", trio, "native"), fused=False),
        Case("rgb libjpeg (k3_jfif)", Entry("", trio, "rgb", LJ), fused=False),
        Case("scaled 1/2 1/4 1/8 (k2_scaled)", Entry("", trio, "yuv_planar", scales=[2, 4, 8]), call="scaled", fused=False),
        Case("resized (k4_resize)", Entry("", trio, "rgb", scales=[1, 2, 1],
                                          resize=([(224, 224), (97, 61), (501, 300)], [api.FILTER_BILINEAR, api.FILTER_LANCZOS, api.FILTER_BICUBIC])),
             call="resized"),
        Case("prepare, run, run", Entry("", trio, "rgb_planar"), call="prepare", fused=True),
        Case("truncated", Entry("", truncated_batch(), "rgb"), status=api.BAD_JPEG, watch=[1]),
        Case("pageable deferred copy", Entry("", big_batch(), "rgb", env={"ROCJPEG_B200_DEFERRED_COPY": "1"}), pageable_deferred=True),
    ]
    for lanes in (1, 4, 8):   # 24 pictures of similar size: every lane gets some; the first and the last lane's pictures
        batch = trio * 8
        C.append(Case(f"{lanes} lanes", Entry("", batch, "rgb_planar", env={"ROCJPEG_B200_LANES": str(lanes)}), watch=[0, len(batch) - 1],
                      lanes=lanes))
    # every destination on device 0: device 1 stores its share there through peer access
    C.append(Case("sharded, destinations on device 0", Entry("", big_batch(), "rgb"), sharded=True, devices=2, dst_device=0))
    # every destination on device 1: the pictures follow their buffers, device 1 decodes them all
    C.append(Case("sharded, destinations on device 1", Entry("", big_batch(), "rgb"), sharded=True, devices=1, dst_device=1))
    return C


CASE_LIST = build_cases()


@pytest.fixture(scope="module")
def oracles(orc):
    return jo.JfifOracle(orc), so.ScaledOracle(orc)


_WANT = {}


def want_of(orc, oracles, case, dec):
    """Whole channel arrays of every picture. A truncated picture's come from the same call with nothing pending (its rows
    before the cut checked against the oracle, as test_handle_history_gpu does)."""
    import torch

    if case.name not in _WANT:
        e = case.entry
        if case.status == api.BAD_JPEG:
            clean = expected(orc, *oracles, Entry("", e.datas[:1], e.fmt))
            t = Target(orc, case)
            torch.cuda.synchronize()
            t.call(dec, t.parse())
            got = t.fetch()
            gu.assert_same(got[0], clean[0], "truncated batch: the clean picture")
            rc, info = orc.parse(e.datas[1])
            head = orc.decode(e.datas[1], "rgb", fill=gu.FILL)[1][0][:112]
            assert np.array_equal(got[1][0][:112, :3 * info.width], head[:, :3 * info.width]), "truncated picture: rows before the cut"
            _WANT[case.name] = got
        else:
            _WANT[case.name] = expected(orc, *oracles, e)
    return _WANT[case.name]


class Target:
    """The destinations of one case: torch buffers (channel + canaries) filled with gu.FILL."""

    def __init__(self, orc, case):
        import torch

        self.case, e = case, case.entry
        self.layout = layout(orc, e)
        with torch.cuda.device(case.dst_device):
            self.bufs = [[torch.full((rows * p + e.mis + 64,), gu.FILL, dtype=torch.uint8, device="cuda") for (rows, _), p in zip(*lay)]
                         for lay in self.layout]
        self.watch = list(range(len(e.datas))) if case.watch is None else case.watch

    def region(self, k, c):
        """Picture k's channel c inside its buffer."""
        (rows, _), p = self.layout[k][0][c], self.layout[k][1][c]
        return self.bufs[k][c][self.case.entry.mis:self.case.entry.mis + rows * p]

    def pattern(self, k, c, size=None):
        """A known pattern P for the whole buffer of picture k's channel c (`size` bytes, default the buffer's), on the
        host: arange % 251 in the channel (no decoded picture looks like it), gu.FILL in the canaries."""
        mis, n = self.case.entry.mis, self.region(k, c).numel()
        out = np.full(size or self.bufs[k][c].numel(), gu.FILL, np.uint8)
        out[mis:mis + n] = np.arange(n) % 251
        return out

    def parse(self):
        with knobs(self.case.entry.env):
            streams = [stream(d) for d in self.case.entry.datas]
        if self.case.pageable_deferred:
            assert not any(s.info().source_is_zero_copy for s in streams)
        return streams

    def dests(self):
        mis = self.case.entry.mis
        return [[(b.data_ptr() + mis, p) for b, p in zip(bufs, lay[1])] for bufs, lay in zip(self.bufs, self.layout)]

    def call(self, dec, streams, run=False):
        """The case's call (run: the Run of a prepared batch). Returns the status."""
        case, e = self.case, self.case.entry
        dec.set_color_convention(e.conv)
        params = api.make_params(e.fmt, e.crop)
        with knobs(e.env):
            if run:
                return dec.run()
            if case.call == "decode":
                return dec.decode(streams[0], params, self.dests()[0])
            if case.call == "scaled":
                return dec.decode_batched_scaled(streams, params, self.dests(), e.scales)
            if case.call == "resized":
                return dec.decode_batched_resized(streams, params, self.dests(), *e.resize, e.scales)
            if case.call == "prepare":
                return dec.prepare(streams, params, self.dests())
            return dec.decode_batched(streams, params, self.dests())

    def fetch(self, bufs=None):
        """Host copies of the whole channel arrays of every picture (of `bufs`, copies of the buffers, if given)."""
        return [gu.fetch(b, lay[1], lay[0], self.case.entry.mis) for b, lay in zip(self.bufs if bufs is None else bufs, self.layout)]


def check_stats(dec, case):
    s = dec.stats()
    if case.fused is not None:
        assert (s.fused_blocks > 0) == case.fused, (case.name, s.fused_blocks)
    if case.lanes is not None:
        assert s.lanes == case.lanes, (case.name, s.lanes)
    if case.devices is not None:
        assert s.devices == case.devices, (case.name, s.devices)


def queue_spin(torch, device):
    """A spin on `device`'s legacy default stream; returns an event right behind it."""
    assert torch.cuda.default_stream(device).cuda_stream == 0, "torch's default stream is not the legacy default stream"
    with torch.cuda.device(device):
        torch.cuda._sleep(SLEEP_CYCLES)
    return event_behind(torch, device)


def event_behind(torch, device):
    with torch.cuda.device(device):
        ev = torch.cuda.Event()
        ev.record()
    return ev


@pytest.fixture(scope="module")
def dec():
    import torch

    assert torch.cuda.is_available()
    torch.cuda.set_device(0)
    d = api.Decoder(api.BACKEND_HARDWARE, 0)
    yield d
    d.close()


@pytest.fixture(scope="module")
def sharded_dec():
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    old = os.environ.get("ROCJPEG_B200_DEVICES")
    os.environ["ROCJPEG_B200_DEVICES"] = "2"
    try:
        d = api.Decoder(api.BACKEND_HARDWARE, 0)
    finally:
        if old is None:
            os.environ.pop("ROCJPEG_B200_DEVICES")
        else:
            os.environ["ROCJPEG_B200_DEVICES"] = old
    if d.num_devices() < 2:
        d.close()
        pytest.skip("no peer access between device 0 and 1")
    yield d
    d.close()


def shard_watch(case):
    """Sharded case with every destination on device 0: the pictures the library's plan gives device 1 (written through
    peer stores)."""
    costs = [stream(d).info().raw_bytes for d in case.entry.datas]
    plan = api.plan_shards(costs, 2)
    watch = [k for k in range(len(costs)) if plan[k] == 1]
    assert watch
    return watch


@pytest.mark.parametrize("hazard", HAZARDS)
@pytest.mark.parametrize("case", CASE_LIST, ids=[re.sub(r"[^0-9a-z]+", "_", c.name.lower()).strip("_") for c in CASE_LIST])
def test_call_is_ordered_after_pending_default_stream_work(request, orc, oracles, case, hazard):
    import torch

    if case.call == "prepare" and hazard == "allocator":
        pytest.skip("a prepared batch's destinations are fixed at Prepare: the allocator idiom cannot hand it a new block")
    d = request.getfixturevalue("sharded_dec" if case.sharded else "dec")
    torch.cuda.set_device(0)
    want = want_of(orc, oracles, case, d)
    pend_dev = case.dst_device
    t = Target(orc, case)
    if case.sharded and case.dst_device == 0:
        t.watch = shard_watch(case)
    # the same call with nothing pending, so that the call under test allocates nothing
    torch.cuda.synchronize()
    st = t.call(d, t.parse())
    assert st == case.status, (case.name, "warm-up", api.STATUS.get(st, st))
    if case.call == "prepare":
        assert t.call(d, None, run=True) == case.status

    calls = 2 if case.call == "prepare" else 1
    streams = t.parse()
    if case.call == "prepare":
        torch.cuda.synchronize()
        assert t.call(d, streams) == api.SUCCESS
    bad = []
    for rep in range(calls):
        # the queued operations once outside the window, so that their kernels are loaded before it
        with torch.cuda.device(pend_dev):
            for k in t.watch:
                for c in range(len(t.bufs[k])):
                    t.region(k, c).fill_(OVERWRITE)
        for bufs in t.bufs:
            for b in bufs:
                b.fill_(gu.FILL)
        k_alloc = t.watch[-1]
        pats, snaps = {}, {}
        if hazard == "write_after_read":
            pats = {(k, c): t.pattern(k, c) for k in t.watch for c in range(len(t.bufs[k]))}
            for (k, c), p in pats.items():
                t.bufs[k][c].copy_(torch.from_numpy(p))
                snaps[(k, c)] = torch.empty_like(t.bufs[k][c])
        if hazard == "allocator":
            # (the pattern is made on the host: no device temporaries of the same size class compete for the freed block)
            torch.cuda.synchronize()
            gc.collect()
            with torch.cuda.device(pend_dev):
                torch.cuda.empty_cache()
                old_contents = t.pattern(k_alloc, 0, max(ALLOC_BYTES, t.bufs[k_alloc][0].numel()))
                x = torch.from_numpy(old_contents).to("cuda")
                reader = torch.empty_like(x)   # allocated here: a new segment in the window would be a cudaMalloc
        torch.cuda.synchronize()

        # the window: nothing in it may synchronise the device (module docstring)
        gc.collect()
        gc.disable()
        try:
            if hazard != "read_after_return":
                ev_spin = queue_spin(torch, pend_dev)
                with torch.cuda.device(pend_dev):
                    if hazard == "write_after_write":
                        for k in t.watch:
                            for c in range(len(t.bufs[k])):
                                t.region(k, c).fill_(OVERWRITE)
                    elif hazard == "write_after_read":
                        for kc, s in snaps.items():
                            s.copy_(t.bufs[kc[0]][kc[1]])
                    else:
                        reader.copy_(x)
                        old = x.data_ptr()
                        del x
                        t.bufs[k_alloc][0] = torch.empty(old_contents.size, dtype=torch.uint8, device="cuda")
                        assert t.bufs[k_alloc][0].data_ptr() == old, "the caching allocator did not hand the freed block on"
                ev_op = event_behind(torch, pend_dev)
                assert not ev_op.query(), "the queued operation finished before the call"
                assert not ev_spin.query(), ("the spin finished before the call: something in the window synchronised the "
                                             "device, or SLEEP_CYCLES is too short")

            st = t.call(d, streams, run=case.call == "prepare")
            if hazard == "read_after_return":
                with torch.cuda.device(pend_dev):
                    copies = [[b.clone() for b in bufs] for bufs in t.bufs]
        finally:
            gc.enable()
        torch.cuda.synchronize()

        what = f"{case.name} {hazard}" + (f" run {rep}" if case.call == "prepare" else "")
        assert st == case.status, (what, api.STATUS.get(st, st))
        check_stats(d, case)
        if hazard == "write_after_read":
            for (k, c), s in snaps.items():
                if not np.array_equal(s.cpu().numpy(), pats[(k, c)]):
                    bad.append(f"{what}: picture {k} channel {c}: the queued copy saw bytes the call wrote")
        if hazard == "allocator" and not np.array_equal(reader.cpu().numpy(), old_contents):
            bad.append(f"{what}: picture {k_alloc}: the queued reader of the freed tensor saw bytes the call wrote")
        try:
            got = t.fetch(copies if hazard == "read_after_return" else None)
        except AssertionError as x:
            bad.append(f"{what}: {x}")
            continue
        for k, (g, w) in enumerate(zip(got, want)):
            try:
                gu.assert_same(g, w, f"{what} picture {k}")
            except AssertionError as x:
                bad.append(str(x))
    assert not bad, "\n".join(bad)


def test_unsplit_call_refuses_a_destination_on_a_peer_device(orc, sharded_dec):
    """A call a two-device handle does not split - one picture, Prepare - writes from the handle's device only, after that
    device's default stream only: a destination on the peer device is refused and left untouched."""
    import torch

    data = load("synth_420_500x375_dri7")
    case = Case("one picture on device 1", Entry("", [data], "rgb"), call="decode", dst_device=1)
    t = Target(orc, case)
    torch.cuda.synchronize()
    assert t.call(sharded_dec, t.parse()) == api.INVALID_PARAMETER
    case.call = "prepare"
    assert t.call(sharded_dec, t.parse()) == api.INVALID_PARAMETER
    for b in t.bufs[0]:
        assert bool((b == gu.FILL).all()), "a refused call wrote its destination"

"""stats().kernel_launches counts the kernels a call actually enqueued (-m gpu): every launcher adds what it launches, so the
counter must equal the number of this library's kernels (rjb::) that torch.profiler's CUDA activity trace records for
the call - on the benchmark batches, on mixed scales, and after a failed CTA-boundary check, where the host re-runs the
synchronisation and everything downstream of it."""
import json
import os

import pytest

from rocjpeg_b200 import api, datagen

import gpu_util as gu
import scaled_oracle as so

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
with open(os.path.join(GOLDEN, "golden.json")) as _f:
    CASES = sorted(json.load(_f)["cases"])


def load(name):
    with open(os.path.join(GOLDEN, name + ".jpg"), "rb") as f:
        return f.read()


@pytest.fixture(scope="module")
def dec():
    import torch

    assert torch.cuda.is_available()
    torch.cuda.set_device(0)
    d = api.Decoder(api.BACKEND_HARDWARE, 0)
    yield d
    d.close()


def _profiled_decode(dec, orc, datas, fmt, scales=None):
    """One batched decode under torch.profiler; returns (status, stats, kernels of this library the trace recorded)."""
    import torch
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile

    streams, dests, keep = [], [], []
    for i, data in enumerate(datas):
        s = api.JpegStream()
        assert s.parse(data) == api.SUCCESS
        rc, info = orc.parse(data)
        if scales is not None:
            info = so.scaled_info(info, scales[i])
        dest, bufs, _, _ = gu.alloc_outputs(orc, info, fmt, (0, 0, 0, 0))
        streams.append(s); dests.append(dest); keep.append(bufs)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        if scales is None:
            st = dec.decode_batched(streams, api.make_params(fmt), dests)
        else:
            st = dec.decode_batched_scaled(streams, api.make_params(fmt), dests, scales)
        torch.cuda.synchronize()
    kernels = [e.name for e in prof.events() if e.device_type == DeviceType.CUDA and "rjb::" in e.name]
    return st, dec.stats(), kernels


def _check(dec, orc, datas, fmt, scales=None):
    st, stats, kernels = _profiled_decode(dec, orc, datas, fmt, scales)
    assert st == api.SUCCESS, api.STATUS.get(st, st)
    assert kernels, "the profiler recorded none of this library's kernels"
    assert stats.kernel_launches == len(kernels), (stats.kernel_launches, sorted(kernels))
    return stats


@pytest.mark.parametrize("lanes", ["1", "4"])
def test_c3(dec, orc, lanes, monkeypatch):
    monkeypatch.setenv("ROCJPEG_B200_LANES", lanes)
    datas, fmt = datagen.workload("c3", 256)
    assert _check(dec, orc, datas, fmt).lanes == int(lanes)


def test_c2(dec, orc):
    datas, fmt = datagen.workload("c2")
    _check(dec, orc, datas, fmt)


@pytest.mark.parametrize("fmt", ["rgb", "yuv_planar"])
def test_mixed_scales(dec, orc, fmt):
    datas = [load(n) for n in CASES]
    _check(dec, orc, datas, fmt, scales=[(1, 2, 4, 8)[i % 4] for i in range(len(datas))])


def test_forced_fallback_after_a_failed_boundary_check(dec, orc, monkeypatch):
    """A one-subsequence halo makes k1_fused's boundary check fail: more k1_sync rounds, then k1_clear_short, k1_write, the DC
    kernels and everything after them."""
    monkeypatch.setenv("ROCJPEG_B200_HALO", "1")
    monkeypatch.setenv("ROCJPEG_B200_SUBSEQ", "32")
    datas = [datagen.make_jpeg(500, 375, css, seed=700 + i) for i, css in enumerate(("444", "422", "420", "444"))]
    assert _check(dec, orc, datas, "rgb_planar").sync_rounds > 1


def test_single_sync_round(dec, orc, monkeypatch):
    """Only round 0 of k1_sync up front: the host runs the rounds the batch still needs, then the downstream stages again."""
    monkeypatch.setenv("ROCJPEG_B200_SYNC_ROUNDS", "1")
    monkeypatch.setenv("ROCJPEG_B200_SUBSEQ", "32")
    assert _check(dec, orc, [load("synth_444_500x375")], "rgb").sync_rounds >= 2

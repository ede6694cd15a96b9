"""Resized decodes (rocJpegB200DecodeBatchedResized) against the plain decode they extend, on workloads of
rocjpeg_b200.datagen:
  c3      256 ImageNet-shaped 500x375 pictures -> 224x224 BILINEAR, RGB_PLANAR, under both colour conventions;
  c2      one 1920x1080 4:2:0 picture -> 224x224 BILINEAR, RGB;
  c4_dri  64 3840x2160 4:2:2 pictures decoded at 1/4 -> 960x540 BICUBIC, RGB, libjpeg convention (exact at that scale).

One JSON line per (workload, convention):
  plain_ms / resized_ms  rocJpegB200Prepare[Scaled|Resized] once, rocJpegB200Run per step, device time of the step (first
                  to last CUDA event); a 256 MiB buffer is written between steps so the L2 holds nothing of the batch. The
                  two calls are measured in alternating rounds; medians over all steps, each round's median beside them.
  resize_passes   k4_resize_h + k4_resize_v on one pipeline lane (CUDA kernel times from torch.profiler), beside the plain
                  decode's output stage on one lane, and the passes' algorithmic bytes - decoded rows read, intermediate rows
                  written and read, output written - over their time as a fraction of 7.7 TB/s.
  cpu_*           what the call replaces on the host: Pillow decode (draft() at the scale), convert, resize, on all threads.
  check           sampled pictures byte for byte: Pillow's resize of the plain decode's output; under the libjpeg convention
                  also the whole Pillow pipeline (decode, draft, resize).
The card's name and power limit are read in the same run. Usage:
  python profiles/bench_resize.py [--workloads c3,c2,c4_dri] [--steps 20] [--warmup 5] [--rounds 3] [--out FILE]
"""
import argparse
import io
import json
import os
import statistics
import sys
import time
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

from bench_scaled import card_context  # noqa: E402

HBM_BYTES_PER_S = 7.7e12   # HGX B200 data sheet, one GPU
# workload -> (output format, scale denominator, (width, height), filter, conventions)
PLANS = {
    "c3": ("rgb_planar", 1, (224, 224), "BILINEAR", ("reference", "libjpeg")),
    "c2": ("rgb", 1, (224, 224), "BILINEAR", ("reference",)),
    "c4_dri": ("rgb", 4, (960, 540), "BICUBIC", ("libjpeg",)),
}
CONVENTIONS = {"reference": 0, "libjpeg": 1}


def pass_bytes(sizes, out_size, filt, ch):
    """Algorithmic bytes of the two passes: the source rows of Pillow's ybox read once, the intermediate rows written and
    read once, the output written."""
    from rocjpeg_b200 import api

    W, H = out_size
    total = 0
    for w, h in sizes:
        if h == H:
            rows = h
        else:
            b, _ = api.resize_coefficients(h, H, filt)
            rows = int(b[-1, 0] + b[-1, 1] - b[0, 0])
        total += rows * w * ch + 2 * rows * W * ch + W * H * ch
    return total


def pillow_pipeline(data, d, mode, size, filt):
    from PIL import Image

    img = Image.open(io.BytesIO(data))
    if d > 1:
        img.draft(mode, (-(-img.size[0] // d), -(-img.size[1] // d)))
    return img.convert(mode).resize(size, filt)


def cpu_baseline(datas, d, mode, size, filt, budget_s):
    threads = os.cpu_count() or 1
    with ThreadPoolExecutor(threads) as ex:
        list(ex.map(lambda x: pillow_pipeline(x, d, mode, size, filt), datas))   # warm-up
        passes, t0 = 0, time.perf_counter()
        while True:
            list(ex.map(lambda x: pillow_pipeline(x, d, mode, size, filt), datas))
            passes += 1
            el = time.perf_counter() - t0
            if el >= budget_s or passes >= 100:
                break
    return 1e3 * el / passes, threads


def kernel_ms(prof, needle):
    total = 0.0
    for e in prof.key_averages():
        if needle in e.key:
            t = getattr(e, "device_time_total", None)
            total += (t if t is not None else e.cuda_time_total) / 1e3
    return total


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="c3,c2,c4_dri")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--cpu-budget", type=float, default=3.0)
    ap.add_argument("--check", type=int, default=8, help="pictures compared with Pillow")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()

    import numpy as np
    import torch
    from PIL import Image
    from torch.profiler import ProfilerActivity, profile

    from rocjpeg_b200 import api, datagen

    assert torch.cuda.is_available(), "bench_resize.py measures the GPU; there is no CPU fallback"
    torch.cuda.set_device(0)
    ctx = card_context(torch)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def l2_flush():
        flush.fill_(1)
        torch.cuda.synchronize()

    for wl in args.workloads.split(","):
        fmt, d, size, filt_name, convs = PLANS[wl]
        filt = getattr(api, "FILTER_" + filt_name)
        pil_filt = getattr(Image, filt_name)
        W, H = size
        ch = 1 if fmt == "y" else 3
        datas, _ = datagen.workload(wl)
        n = len(datas)
        dec = api.Decoder(api.BACKEND_HARDWARE, 0)
        offs, total = [], 0
        for x in datas:
            offs.append(total)
            total += (len(x) + 63) // 64 * 64
        arena = torch.empty(total + 64, dtype=torch.uint8, pin_memory=True)
        an = arena.numpy()
        for o, x in zip(offs, datas):
            an[o:o + len(x)] = memoryview(x)
        streams = []
        for o, x in zip(offs, datas):
            s = api.JpegStream()
            assert s.parse_ptr(arena.data_ptr() + o, len(x), arena) == api.SUCCESS
            streams.append(s)
        # plain decode at 1/d (its own buffers) and the resized call (W x H buffers)
        plain_dests, plain_keep, sizes = [], [], []
        for s in streams:
            _, css, ws, hs = dec.scaled_image_info(s, d)
            w, h = ws[0], hs[0]
            sizes.append((w, h))
            chans = api.output_channel_shapes(api.CSS_NAME[css], fmt, w, h)
            pitch = chans[0][1]
            bufs = [torch.empty(rows * pitch + 64, dtype=torch.uint8, device="cuda") for rows, _ in chans]
            plain_keep.append((bufs, pitch, w, h))
            plain_dests.append([(b.data_ptr(), pitch) for b in bufs])
        rchans = api.output_channel_shapes("444", fmt, W, H)
        rpitch = rchans[0][1]
        rkeep = [[torch.empty(rows * rpitch + 64, dtype=torch.uint8, device="cuda") for rows, _ in rchans] for _ in streams]
        rdests = [[(b.data_ptr(), rpitch) for b in bufs] for bufs in rkeep]
        params = api.make_params(fmt)
        scales = [d] * n

        def prepare(kind):
            if kind == "plain":
                return dec.prepare(streams, params, plain_dests, scales)
            return dec.prepare_resized(streams, params, rdests, [size] * n, filt, scales)

        def fetch(bufs, pitch, w, h):
            chans = [b.cpu().numpy()[:h * pitch].reshape(h, pitch) for b in bufs]
            if fmt == "rgb":
                return chans[0][:, :3 * w].reshape(h, w, 3)
            return np.stack([c[:, :w] for c in chans], -1) if fmt == "rgb_planar" else chans[0][:, :w]

        for c in convs:
            dec.set_color_convention(CONVENTIONS[c])
            res = {k: {"steps": [], "rounds": []} for k in ("plain", "resized")}
            dec.set_profiling(2)
            for _ in range(args.rounds):
                for kind in ("plain", "resized"):
                    assert prepare(kind) == api.SUCCESS
                    for _ in range(args.warmup):
                        assert dec.run() == api.SUCCESS
                    ms = []
                    for _ in range(args.steps):
                        l2_flush()
                        assert dec.run() == api.SUCCESS
                        ms.append(dec.stats().total_ms)
                    res[kind]["steps"] += ms
                    res[kind]["rounds"].append(statistics.median(ms))
                    res[kind]["launches"] = dec.stats().kernel_launches
                    res[kind]["lanes"] = dec.stats().lanes
            # byte checks: the resized output against Pillow's resize of the plain decode (and the Pillow pipeline)
            dec.set_profiling(0)
            assert prepare("plain") == api.SUCCESS and dec.run() == api.SUCCESS
            picks = sorted({int(k) for k in np.linspace(0, n - 1, min(args.check, n))})
            src = {k: fetch(*plain_keep[k]) for k in picks}
            assert prepare("resized") == api.SUCCESS and dec.run() == api.SUCCESS
            torch.cuda.synchronize()
            mode = "L" if fmt == "y" else "RGB"
            pipeline_equal = 0
            for k in picks:
                got = fetch(rkeep[k], rpitch, W, H)
                want = np.asarray(Image.fromarray(src[k]).resize(size, pil_filt))
                assert np.array_equal(got, want), f"{wl} {c} picture {k} differs from Pillow's resize of the plain decode"
                if c == "libjpeg":
                    pil = np.asarray(pillow_pipeline(datas[k], d, mode, size, pil_filt))
                    assert np.array_equal(got, pil), f"{wl} picture {k} differs from the Pillow pipeline"
                    pipeline_equal += 1
            # one lane: the passes' kernel times, and the plain decode's output stage for scale
            os.environ["ROCJPEG_B200_LANES"] = "1"
            dec.set_profiling(1)
            stage = {}
            for kind in ("plain", "resized"):
                assert prepare(kind) == api.SUCCESS
                for _ in range(3):
                    assert dec.run() == api.SUCCESS
                k_steps = max(3, min(args.steps, 10))
                acc = 0.0
                for _ in range(k_steps):
                    l2_flush()
                    assert dec.run() == api.SUCCESS
                    acc += dec.stats().stage_ms[api.STAGES.index("output")]
                stage[kind] = acc / k_steps
            dec.set_profiling(0)
            k_steps = max(3, min(args.steps, 10))
            l2_flush()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(k_steps):
                    assert dec.run() == api.SUCCESS
                torch.cuda.synchronize()
            h_ms, v_ms = kernel_ms(prof, "k4_resize_h") / k_steps, kernel_ms(prof, "k4_resize_v") / k_steps
            del os.environ["ROCJPEG_B200_LANES"]
            nbytes = pass_bytes(sizes, size, filt, ch)
            cpu_ms, threads = cpu_baseline(datas, d, mode, size, pil_filt, args.cpu_budget)
            pm, rm = statistics.median(res["plain"]["steps"]), statistics.median(res["resized"]["steps"])
            line = {
                "workload": wl, "convention": c, "output_format": fmt, "scale_denom": d, "size": list(size), "filter": filt_name,
                "batch": n, **ctx,
                "plain_ms": round(pm, 4), "resized_ms": round(rm, 4),
                "plain_round_medians_ms": [round(x, 4) for x in res["plain"]["rounds"]],
                "resized_round_medians_ms": [round(x, 4) for x in res["resized"]["rounds"]],
                "steps": len(res["plain"]["steps"]), "lanes": res["resized"]["lanes"],
                "kernel_launches": {"plain": res["plain"]["launches"], "resized": res["resized"]["launches"]},
                "resize_passes": {"k4_resize_h_ms": round(h_ms, 4), "k4_resize_v_ms": round(v_ms, 4),
                                  "output_stage_ms_one_lane": {"plain": round(stage["plain"], 4), "resized": round(stage["resized"], 4)},
                                  "algorithmic_bytes": nbytes,
                                  "hbm_fraction": round(nbytes / ((h_ms + v_ms) * 1e-3) / HBM_BYTES_PER_S, 3) if h_ms + v_ms > 0 else None},
                "cpu_pillow_ms": round(cpu_ms, 3), "cpu_threads": threads,
                "check": f"{len(picks)} pictures equal Pillow's resize of the plain decode"
                         + (f"; {pipeline_equal} equal Pillow's decode{' + draft' if d > 1 else ''} + resize" if c == "libjpeg" else ""),
                "l2": "256 MiB device buffer written between timed steps",
            }
            text = json.dumps(line)
            print(text, flush=True)
            if args.out:
                with open(args.out, "a") as f:
                    f.write(text + "\n")
        dec.close()


if __name__ == "__main__":
    main()

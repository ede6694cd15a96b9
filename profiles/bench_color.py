"""The two colour conventions of RGB / RGB_PLANAR against each other, on the workloads c3 (256 ImageNet-shaped 500x375
pictures, 4:4:4 / 4:2:2 / 4:2:0 -> RGB_PLANAR) and c2 (one 1920x1080 4:2:0 picture -> RGB) of rocjpeg_b200.datagen.
The reference convention runs the fused IDCT + colour kernel on whole pictures; the libjpeg convention runs the IDCT into
the plane arena and then k3_jfif, so it is expected to be slower there.

One JSON line per (workload, convention):
  resident_ms     rocJpegB200Prepare once, rocJpegB200Run per step, device time of the step (first to last CUDA event); a
                  256 MiB buffer is written between steps so the L2 holds nothing of the batch. The conventions are measured
                  in alternating rounds; the median over all steps is reported, each round's median beside it.
  stage_ms        a separate pass with per-stage events (profiling level 1) on one pipeline lane.
  output_stage    (libjpeg only) the output stage of that pass (k3_jfif, one launch) and its algorithmic HBM traffic: plane
                  bytes read (each 256 x 32 tile's luma and its chroma with the one-sample halo fancy upsampling reads) plus
                  pixels written, over its time, as a fraction of 7.7 TB/s.
  cpu_*           libjpeg-turbo's default decode to RGB (the libjpeg convention's output) on all host threads.
  check           pictures of the batch compared byte for byte: libjpeg convention with libjpeg-turbo.
The card's name and power limit are read in the same run. Usage:
  python profiles/bench_color.py [--workloads c3,c2] [--steps 20] [--warmup 5] [--rounds 3] [--out FILE]
"""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

from bench_scaled import card_context  # noqa: E402

HBM_BYTES_PER_S = 7.7e12   # HGX B200 data sheet, one GPU
CONVENTIONS = {"reference": 0, "libjpeg": 1}


def k3_jfif_bytes(infos):
    """Algorithmic bytes of k3_jfif over a batch: per 256 x 32 output tile the luma it reads, each chroma plane's samples
    under it plus the one-sample halo of fancy upsampling (clamped to the picture), and the three bytes per pixel it writes."""
    total = 0
    for w, h, sx, sy in infos:
        cw, ch = -(-w // (1 << sx)), -(-h // (1 << sy))
        for ty in range(0, h, 32):
            th = min(32, h - ty)
            r0, r1 = max(0, (ty >> sy) - 1), min(ch, ((ty + th - 1) >> sy) + 2)
            for tx in range(0, w, 256):
                tw = min(256, w - tx)
                c0, c1 = max(0, (tx >> sx) - 1), min(cw, ((tx + tw - 1) >> sx) + 2)
                total += tw * th * 4 + 2 * (r1 - r0) * (c1 - c0)
    return total


def cpu_baseline(datas, budget_s):
    import numpy as np

    import oracle

    ljt, orc = oracle.LibJpegTurbo(), oracle.Oracle()
    threads = os.cpu_count() or 1
    outs, pitches = [], []
    for x in datas:
        rc, i = orc.parse(x)
        outs.append(np.empty((i.height, i.width * 3), np.uint8))
        pitches.append(i.width * 3)
    ljt.decode_batch(datas, outs, pitches, 0, threads)   # warm-up
    passes, t0 = 0, time.perf_counter()
    while True:
        ljt.decode_batch(datas, outs, pitches, 0, threads)
        passes += 1
        el = time.perf_counter() - t0
        if el >= budget_s or passes >= 200:
            break
    return {"cpu_ms_per_batch": 1e3 * el / passes, "cpu_threads": threads, "cpu_passes": passes}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="c3,c2")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--cpu-budget", type=float, default=3.0)
    ap.add_argument("--check", type=int, default=8, help="pictures compared with libjpeg-turbo")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()

    import numpy as np
    import torch

    import oracle
    from rocjpeg_b200 import api, datagen

    assert torch.cuda.is_available(), "bench_color.py measures the GPU; there is no CPU fallback"
    torch.cuda.set_device(0)
    ctx = card_context(torch)
    ljt = oracle.LibJpegTurbo()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def l2_flush():
        flush.fill_(1)
        torch.cuda.synchronize()

    for wl in args.workloads.split(","):
        datas, fmt = datagen.workload(wl)
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
        infos, dests, keep, px = [], [], [], 0
        for s in streams:
            i = s.info()
            css = api.CSS_NAME[i.chroma_subsampling]
            px += i.width * i.height
            infos.append((i.width, i.height, 1 if css in ("422", "420") else 2 if css == "411" else 0, 1 if css in ("440", "420") else 0))
            chans = api.output_channel_shapes(css, fmt, i.width, i.height)
            pitch = chans[0][1]
            bufs = [torch.empty(rows * pitch + 64, dtype=torch.uint8, device="cuda") for rows, _ in chans]
            keep.append((bufs, pitch, i.width, i.height))
            dests.append([(b.data_ptr(), pitch) for b in bufs])
        params = api.make_params(fmt)
        res = {c: {"steps": [], "rounds": []} for c in CONVENTIONS}

        dec.set_profiling(2)
        for r in range(args.rounds):
            for c, conv in CONVENTIONS.items():
                dec.set_color_convention(conv)
                assert dec.prepare(streams, params, dests) == api.SUCCESS
                for _ in range(args.warmup):
                    assert dec.run() == api.SUCCESS
                ms = []
                for _ in range(args.steps):
                    l2_flush()
                    assert dec.run() == api.SUCCESS
                    ms.append(dec.stats().total_ms)
                res[c]["steps"] += ms
                res[c]["rounds"].append(statistics.median(ms))
                res[c]["launches"] = dec.stats().kernel_launches
                res[c]["fused_blocks"] = dec.stats().fused_blocks
        # the libjpeg convention's output against libjpeg-turbo's default decode
        dec.set_color_convention(CONVENTIONS["libjpeg"])
        assert dec.prepare(streams, params, dests) == api.SUCCESS
        assert dec.run() == api.SUCCESS
        torch.cuda.synchronize()
        picks = sorted({int(k) for k in np.linspace(0, n - 1, min(args.check, n))})
        for k in picks:
            bufs, pitch, w, h = keep[k]
            want = ljt.decode_rgb(datas[k], w, h)
            chans = [b.cpu().numpy()[:h * pitch].reshape(h, pitch) for b in bufs]
            got = chans[0][:, :3 * w].reshape(h, w, 3) if fmt == "rgb" else np.stack([ch[:, :w] for ch in chans], -1)
            assert np.array_equal(got, want), f"{wl} picture {k} differs from libjpeg-turbo"
        # per-stage times: one lane, an event after every stage
        os.environ["ROCJPEG_B200_LANES"] = "1"
        dec.set_profiling(1)
        for c, conv in CONVENTIONS.items():
            dec.set_color_convention(conv)
            assert dec.prepare(streams, params, dests) == api.SUCCESS
            for _ in range(3):
                assert dec.run() == api.SUCCESS
            acc = [0.0] * len(api.STAGES)
            k = max(3, min(args.steps, 10))
            for _ in range(k):
                l2_flush()
                assert dec.run() == api.SUCCESS
                st = dec.stats()
                for i in range(len(api.STAGES)):
                    acc[i] += st.stage_ms[i]
            res[c]["stage_ms"] = {name: round(v / k, 4) for name, v in zip(api.STAGES, acc)}
        del os.environ["ROCJPEG_B200_LANES"]
        dec.set_profiling(0)
        cpu = cpu_baseline(datas, args.cpu_budget)
        jb = k3_jfif_bytes(infos)
        for c in CONVENTIONS:
            r = res[c]
            ms = statistics.median(r["steps"])
            line = {
                "workload": wl, "convention": c, "output_format": fmt, "batch": n, **ctx,
                "resident_ms": round(ms, 4), "resident_round_medians_ms": [round(x, 4) for x in r["rounds"]],
                "resident_steps": len(r["steps"]), "kernel_launches": r["launches"], "fused_blocks": r["fused_blocks"],
                "resident_mp_per_s": round(px / ms / 1e3, 1), "stage_ms_one_lane": r["stage_ms"],
                "cpu_libjpeg_turbo_ms": round(cpu["cpu_ms_per_batch"], 3), "cpu_threads": cpu["cpu_threads"],
                "cpu_mp_per_s": round(px / cpu["cpu_ms_per_batch"] / 1e3, 1),
                "l2": "256 MiB device buffer written between timed steps",
            }
            if c == "libjpeg":
                out_ms = r["stage_ms"]["output"]
                line["output_stage"] = {"kernel": "k3_jfif", "ms_one_lane": out_ms, "algorithmic_bytes": jb,
                                        "hbm_fraction": round(jb / (out_ms * 1e-3) / HBM_BYTES_PER_S, 3) if out_ms > 0 else None}
                line["check"] = f"{len(picks)} pictures equal libjpeg-turbo's default decode"
            text = json.dumps(line)
            print(text, flush=True)
            if args.out:
                with open(args.out, "a") as f:
                    f.write(text + "\n")
        dec.close()


if __name__ == "__main__":
    main()

"""Decodes at 1/2, 1/4 and 1/8 scale against full size, on the workloads c3 (256 ImageNet-shaped 500x375 pictures ->
RGB_PLANAR) and c4_dri (64 x 3840x2160 4:2:2 with restart markers -> YUV_PLANAR) of rocjpeg_b200.datagen.

One JSON line per (workload, scale denominator):
  resident_ms    rocJpegB200PrepareScaled once, then rocJpegB200Run per step, device time of the step (first to last CUDA
                 event); a 256 MiB buffer is written between steps so the L2 holds nothing of the batch. The scales are
                 measured in alternating rounds; the median over all steps is reported, each round's median beside it.
  e2e_ms         rocJpegB200DecodeBatchedScaled, wall clock of the call, files in page-locked host memory (parsed once).
  stage_ms       a separate pass with per-stage events (profiling level 1) on one pipeline lane.
  cpu_*          libjpeg-turbo at the same scale (scale_denom d, its default decode) on all host threads.
  rates          images/s and MP/s, counting source pixels (W x H) and output pixels (ceil(W/d) x ceil(H/d)).
  check          pictures of the last resident step compared byte for byte with the oracle.
The card's name and power limit are read in the same run. Usage:
  python profiles/bench_scaled.py [--workloads c3,c4_dri] [--scales 1,2,4,8] [--steps 20] [--warmup 5] [--rounds 3] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))   # scaled_oracle: the oracle and libjpeg-turbo at scale 1/d


def card_context(torch):
    name = torch.cuda.get_device_name(0)
    power = None
    try:
        r = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=20)
        if r.returncode == 0:
            pl, clk = [x.strip() for x in r.stdout.strip().split(",")]
            power = {"power_limit_w": float(pl), "max_sm_clock_mhz": float(clk)}
    except (OSError, ValueError, subprocess.TimeoutExpired):
        pass
    return {"card": name, **(power or {"power_limit_w": None})}


def cpu_baseline(datas, fmt, d, budget_s):
    import numpy as np

    import oracle
    import scaled_oracle

    ljt, orc = scaled_oracle.ScaledLibJpegTurbo(), oracle.Oracle()
    threads = os.cpu_count() or 1
    mode = 0 if fmt in ("rgb", "rgb_planar") else 2
    outs, pitches = [], []
    for x in datas:
        rc, i = orc.parse(x)
        if mode == 0:
            w, h = -(-i.width // d), -(-i.height // d)
            outs.append(np.empty((h, w * 3), np.uint8))
            pitches.append(w * 3)
        else:
            outs.append(np.empty(sum(i.blocks_w[c] * i.blocks_h[c] * 64 for c in range(i.ncomp)), np.uint8))
            pitches.append(0)
    ljt.decode_batch_scaled(datas, outs, pitches, mode, threads, d)   # warm-up
    passes, t0 = 0, time.perf_counter()
    while True:
        ljt.decode_batch_scaled(datas, outs, pitches, mode, threads, d)
        passes += 1
        el = time.perf_counter() - t0
        if el >= budget_s or passes >= 100:
            break
    return {"cpu_ms_per_batch": 1e3 * el / passes, "cpu_threads": threads, "cpu_passes": passes,
            "cpu_output": "RGB" if mode == 0 else "raw YCbCr planes"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="c3,c4_dri")
    ap.add_argument("--scales", default="1,2,4,8")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--cpu-budget", type=float, default=3.0)
    ap.add_argument("--check", type=int, default=3, help="pictures of the last resident step compared with the oracle")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()

    import numpy as np
    import torch

    import oracle
    import scaled_oracle
    from rocjpeg_b200 import api, datagen

    assert torch.cuda.is_available(), "bench_scaled.py measures the GPU; there is no CPU fallback"
    torch.cuda.set_device(0)
    ctx = card_context(torch)
    scales = [int(x) for x in args.scales.split(",")]
    orc = scaled_oracle.ScaledOracle(oracle.Oracle())
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
        src_px = sum(s.info().width * s.info().height for s in streams)
        per_scale = {}
        for d in scales:   # destinations at the scaled size
            dests, keep, out_px = [], [], 0
            for s in streams:
                i = s.info()
                w, h = -(-i.width // d), -(-i.height // d)
                out_px += w * h
                chans = api.output_channel_shapes(api.CSS_NAME[i.chroma_subsampling], fmt, w, h)
                pitches = [rb for (_, rb) in chans]
                if fmt == "yuv_planar" and api.CSS_NAME[i.chroma_subsampling] in ("422", "420"):
                    pitches[2] = pitches[1]
                bufs = [torch.empty(rows * p + 64, dtype=torch.uint8, device="cuda") for (rows, _), p in zip(chans, pitches)]
                keep.append((bufs, pitches, chans))
                dests.append([(b.data_ptr(), p) for b, p in zip(bufs, pitches)])
            per_scale[d] = {"dests": dests, "keep": keep, "out_px": out_px, "steps": [], "rounds": []}
        params = api.make_params(fmt)

        # resident: alternating rounds over the scales
        dec.set_profiling(2)
        for r in range(args.rounds):
            for d in scales:
                ps = per_scale[d]
                assert dec.prepare(streams, params, ps["dests"], [d] * n) == api.SUCCESS
                for _ in range(args.warmup):
                    assert dec.run() == api.SUCCESS
                ms = []
                for _ in range(args.steps):
                    l2_flush()
                    assert dec.run() == api.SUCCESS
                    ms.append(dec.stats().total_ms)
                ps["steps"] += ms
                ps["rounds"].append(statistics.median(ms))
                ps["launches"] = dec.stats().kernel_launches
        # correctness of the last step of each scale: re-run it, compare a sample of pictures with the oracle
        for d in scales:
            ps = per_scale[d]
            assert dec.prepare(streams, params, ps["dests"], [d] * n) == api.SUCCESS
            assert dec.run() == api.SUCCESS
            torch.cuda.synchronize()
            picks = sorted({int(k) for k in np.linspace(0, n - 1, min(args.check, n))})
            for k in picks:
                bufs, pitches, chans = ps["keep"][k]
                _, want = orc.decode_scaled(datas[k], d, fmt, pitches=pitches)
                for b, p, (rows, rb), w in zip(bufs, pitches, chans, want):
                    got = b.cpu().numpy()[:rows * p].reshape(rows, p)
                    assert np.array_equal(got[:, :rb], w[:rows, :rb]), f"{wl} 1/{d} picture {k} differs from the oracle"
            ps["checked"] = len(picks)
        # per-stage times: one lane, an event after every stage
        os.environ["ROCJPEG_B200_LANES"] = "1"
        dec.set_profiling(1)
        for d in scales:
            ps = per_scale[d]
            assert dec.prepare(streams, params, ps["dests"], [d] * n) == api.SUCCESS
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
            ps["stage_ms"] = {name: round(v / k, 4) for name, v in zip(api.STAGES, acc)}
        del os.environ["ROCJPEG_B200_LANES"]
        # end to end: the public scaled call, files in page-locked memory
        dec.set_profiling(0)
        for d in scales:
            ps = per_scale[d]
            batch = dec.make_batch(streams, ps["dests"])
            sc = dec._scales([d] * n, n)
            for _ in range(args.warmup):
                assert dec.decode_batched_scaled(batch, params, None, sc) == api.SUCCESS
            ts = []
            for _ in range(args.steps):
                l2_flush()
                t0 = time.perf_counter()
                rc = dec.decode_batched_scaled(batch, params, None, sc)
                ts.append(time.perf_counter() - t0)
                assert rc == api.SUCCESS
            ps["e2e_ms"] = 1e3 * statistics.median(ts)
        for d in scales:
            ps = per_scale[d]
            res_ms = statistics.median(ps["steps"])
            cpu = cpu_baseline(datas, fmt, d, args.cpu_budget)
            line = {
                "workload": wl, "scale_denom": d, "output_format": fmt, "batch": n, **ctx,
                "resident_ms": round(res_ms, 4), "resident_round_medians_ms": [round(x, 4) for x in ps["rounds"]],
                "resident_steps": len(ps["steps"]), "kernel_launches": ps["launches"],
                "e2e_ms": round(ps["e2e_ms"], 4), "stage_ms": ps["stage_ms"],
                "source_mpixels": round(src_px / 1e6, 3), "output_mpixels": round(ps["out_px"] / 1e6, 3),
                "resident_images_per_s": round(n / res_ms * 1e3, 1),
                "resident_source_mp_per_s": round(src_px / res_ms / 1e3, 1),
                "resident_output_mp_per_s": round(ps["out_px"] / res_ms / 1e3, 1),
                "e2e_images_per_s": round(n / ps["e2e_ms"] * 1e3, 1),
                "e2e_source_mp_per_s": round(src_px / ps["e2e_ms"] / 1e3, 1),
                "cpu_images_per_s": round(n / cpu["cpu_ms_per_batch"] * 1e3, 1),
                "cpu_source_mp_per_s": round(src_px / cpu["cpu_ms_per_batch"] / 1e3, 1),
                **{k: (round(v, 3) if isinstance(v, float) else v) for k, v in cpu.items()},
                "l2": "256 MiB device buffer written between timed steps",
                "check": f"{ps['checked']} pictures of the batch equal the oracle",
            }
            text = json.dumps(line)
            print(text, flush=True)
            if args.out:
                with open(args.out, "a") as f:
                    f.write(text + "\n")
        dec.close()


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""bench.py — decoded MP/s and images/s of rocJpegDecodeBatched on B200 (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c3] [--impl reference] [--dump-outputs DIR]

A "step" is one rocJpegDecodeBatched pass over one batch of synthetic JPEGs (seeded, encoded
here at quality 90 — rocjpeg_b200/datagen.py). Default workload = BASELINE.json configs[2]
("c3": 256 ImageNet-shaped 500x375 images, mixed 4:4:4/4:2:2/4:2:0, -> RGB_PLANAR), the
configuration the metric "rocJpegDecodeBatched at 1/2/4/8 B200" is quoted on; the other
configs are selectable with --workload (c2, c3j, c4_dri, c4_nodri, c5_400, c5_440).

Our arm prints ONE JSON line:
  value        device-resident throughput: batch already in HBM (rocJpegB200Prepare), each step
               = rocJpegB200Run (every kernel of the path), CUDA events on the decoder's stream
  e2e          the same metric through rocJpegDecodeBatched itself: HOST JPEG buffers in, the
               host->device copy of descriptors + entropy-coded bytes and the device->host
               read-back of the decoder's status counters inside the timed region (wall clock
               around the synchronous call, as the reference's samples time it). Pixels stay in
               device memory: that is the API's contract (api/rocjpeg.h:104-107).
  roofline     the dominant kernel stage (by device time) against the measured HBM peak
  cpu_baseline multithreaded libjpeg-turbo (Pillow's 3.1.4.1) decoding the identical files on
               this box's host cores — the baseline BASELINE.json prescribes, because the
               reference has no CPU decode path (src/rocjpeg_decoder.cpp:87-88)
`--impl reference` times that CPU baseline alone and prints it in the same shape.
`--dump-outputs DIR` writes the pixels the last timed step of `value` decoded (the inputs are seeded: the same arguments
decode the same files), so that two builds can be compared output for output.
Multi-GPU: one process per GPU (torchrun), every rank decodes its own full batch (weak
scaling, images are independent — no data-path collective); time = max over ranks.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "decoded_MP_per_s_rocJpegDecodeBatched"
UNIT = "MP/s"
DUMP_BYTES = 56 << 20   # float32 pixels of --dump-outputs: with the row indices and the .npy headers the files stay under 64 MB
WORKLOAD_DESC = {
    "c2": "single 1920x1080 4:2:0 q90 baseline JPEG, no DRI -> RGB (BASELINE configs[1])",
    "c3": "256 x 500x375 q90 baseline JPEGs, 4:4:4/4:2:2/4:2:0 round-robin, no DRI -> RGB_PLANAR (BASELINE configs[2])",
    "c3j": "256 jittered-size (300-640 x 224-500) q90 JPEGs, mixed subsampling -> RGB_PLANAR",
    "c4_dri": "64 x 3840x2160 4:2:2 q90, DRI = one MCU row -> YUV_PLANAR (BASELINE configs[3])",
    "c4_nodri": "64 x 3840x2160 4:2:2 q90, no restart markers -> YUV_PLANAR (BASELINE configs[3])",
    "c5_400": "single 8192x8192 4:0:0 q90, no DRI -> Y (BASELINE configs[4])",
    "c5_440": "single 8192x8192 4:4:0 q90, no DRI -> NATIVE (BASELINE configs[4])",
}


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region: NVML polled from a thread every
    couple of milliseconds (the timed region of the default run is tens of milliseconds, shorter
    than one `nvidia-smi -lms` period); nvidia-smi is the fallback when NVML cannot be loaded."""

    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        self.index = index
        self.sm, self.reasons, self.mx = [], set(), 0
        self.stop_flag = threading.Event()
        self.thread = None
        self.source = None

    def _nvml_loop(self):
        import pynvml as nv

        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(self.index)
        self.mx = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
        bits = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown, "hw_thermal_slowdown": nv.nvmlClocksEventReasonHwThermalSlowdown,
                "sw_thermal_slowdown": nv.nvmlClocksEventReasonSwThermalSlowdown, "sw_power_cap": nv.nvmlClocksEventReasonSwPowerCap}
        self.source = "nvml"
        self.ready.set()
        while not self.stop_flag.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                for n, b in bits.items():
                    if r & b:
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.002)

    def _smi_loop(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        self.source = "nvidia-smi"
        self.ready.set()
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=10).stdout.strip().splitlines()[0]
                f = [x.strip() for x in out.split(",")]
                self.sm.append(float(f[0]))
                self.mx = max(self.mx, float(f[1]))
                for n, v in zip(self.NAMES, f[2:6]):
                    if v.lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                time.sleep(0.05)

    def _loop(self):
        try:
            self._nvml_loop()
        except Exception:
            self._smi_loop()

    def start(self):
        self.ready = threading.Event()
        self.thread = threading.Thread(target=self._loop, daemon=True)
        self.thread.start()
        self.ready.wait(20)
        self.sm.clear()   # keep only samples taken after start() returned

    def stop(self):
        self.stop_flag.set()
        if self.thread:
            self.thread.join(15)
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.mx or None, "reasons": sorted(self.reasons),
                "samples": len(sm), "source": self.source}


def measured_traffic(workload, stage):
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) of a stage's kernel from the
    committed `ncu --set full` capture of this workload (profiles/traffic.json, written by
    profiles/summarize.py); None when no capture of that workload/kernel has been committed."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f)
        return t.get(workload, {}).get(stage)
    except Exception:
        return None


def build_workload(name, n):
    from rocjpeg_b200 import datagen

    datas, fmt = datagen.workload(name, n)
    return datas, fmt


def pixels_of(datas):
    """Total pixels and (width, height, subsampling) per picture, from the library's own parser."""
    from rocjpeg_b200 import api

    tot, dims = 0, []
    s = api.JpegStream()
    for d in datas:
        assert s.parse(d) == api.SUCCESS
        i = s.info()
        tot += i.width * i.height
        dims.append((i.width, i.height, api.CSS_NAME[i.chroma_subsampling]))
    s.close()
    return tot, dims


def run_cpu_baseline(datas, fmt, budget_s=12.0, threads=None):
    """Multithreaded libjpeg-turbo (default islow decode) of the same files, in host memory.
    Returns (MP/s, images/s, threads, description of the sample)."""
    import numpy as np

    import oracle

    ljt = oracle.LibJpegTurbo()
    orc = oracle.Oracle()
    threads = threads or os.cpu_count() or 1
    mode = {"rgb": 0, "rgb_planar": 0, "y": 1, "yuv_planar": 2, "native": 2}[fmt]
    outs, pitches, mp = [], [], 0
    uniq = {}
    for d in datas:
        rc, i = orc.parse(d)
        mp += i.width * i.height
        if mode == 0:
            outs.append(np.empty((i.height, i.width * 3), np.uint8)); pitches.append(i.width * 3)
        elif mode == 1:
            outs.append(np.empty((i.height, i.width), np.uint8)); pitches.append(i.width)
        else:
            n = sum(i.blocks_w[c] * i.blocks_h[c] * 64 for c in range(i.ncomp))
            outs.append(np.empty(n, np.uint8)); pitches.append(0)
    ljt.decode_batch(datas, outs, pitches, mode, threads)   # warm-up pass
    passes, t0 = 0, time.perf_counter()
    while True:
        ljt.decode_batch(datas, outs, pitches, mode, threads)
        passes += 1
        el = time.perf_counter() - t0
        if el >= budget_s or passes >= 200:
            break
    sample = f"{passes} passes over the full batch ({len(datas)} images, {mp / 1e6:.1f} MP) with {threads} host threads, " \
             f"libjpeg-turbo {os.path.basename(ljt.path)} default decode -> " \
             f"{'RGB' if mode == 0 else 'Y' if mode == 1 else 'raw YCbCr planes'} in host memory"
    return mp * passes / el / 1e6, len(datas) * passes / el, threads, sample


def sample_outputs(torch, keep):
    """The valid rows x bytes of every output channel of every picture, copied to the host as uint8: (name, pixels, rows kept).
    When the batch holds more than DUMP_BYTES / 4 samples, each channel keeps the same share of its rows, chosen by a fixed
    seed (rows kept = their indices, else None): the same arguments give the same rows, so two builds of the library can be
    compared output for output."""
    import numpy as np

    total = sum(rows * rb for _, _, chans in keep for rows, rb in chans)
    share = min(1.0, DUMP_BYTES / 4 / total)
    rng = np.random.default_rng(0)
    out = []
    for i, (bufs, pitches, chans) in enumerate(keep):
        for c, (b, p, (rows, rb)) in enumerate(zip(bufs, pitches, chans)):
            plane, kept = b[:rows * p].view(rows, p)[:, :rb], None
            if share < 1.0:
                kept = np.sort(rng.choice(rows, max(1, int(rows * share)), replace=False))
                plane = plane[torch.from_numpy(kept).to(plane.device)]
            out.append((f"image{i:04d}_ch{c}", plane.cpu().numpy(), kept))
    return out


def write_outputs(path, arrays):
    """<name>.npy = the pixels; where rows were sampled, <name>_rows.npy = the index of each of them in the channel."""
    import numpy as np

    os.makedirs(path, exist_ok=True)
    for name, a, kept in arrays:
        np.save(os.path.join(path, name + ".npy"), a.astype(np.float32))
        if kept is not None:
            np.save(os.path.join(path, name + "_rows.npy"), kept.astype(np.float32))


def measure_inlib(api, torch, workload, args, ndev, dev0, ready):
    """One parse + rocJpegDecodeBatched per step, sharded by the library over `ndev` GPUs (ROCJPEG_B200_DEVICES); see main().
    `ready` = the already built single-GPU objects of the same workload (or None: build them, incl. the 1-GPU time)."""
    import numpy as np

    import oracle

    if ready is None:
        datas, fmt = build_workload(workload, args.batch or None)
        _, dims = pixels_of(datas)
        offs, total = [], 0
        for d in datas:
            offs.append(total)
            total += (len(d) + 63) // 64 * 64
        arena = torch.empty(total + 64, dtype=torch.uint8, pin_memory=True)
        an = arena.numpy()
        for o, d in zip(offs, datas):
            an[o:o + len(d)] = memoryview(d)
        addrs, lens, dests0, single_ms = [arena.data_ptr() + o for o in offs], [len(d) for d in datas], None, None
    else:
        datas, fmt, dims, addrs, lens, arena, dests0, single_ms = ready
    total_px = sum(w * h for (w, h, _) in dims)
    params = api.make_params(fmt)

    def alloc(devices):
        dests, keep = [], []
        for (w, h, css), dv in zip(dims, devices):
            chans = api.output_channel_shapes(css, fmt, w, h)
            pitches = [rb for (_, rb) in chans]
            if fmt == "yuv_planar" and css in ("422", "420"):
                pitches[2] = pitches[1]
            bufs = [torch.zeros(rows * p + 64, dtype=torch.uint8, device=f"cuda:{dv}") for (rows, _), p in zip(chans, pitches)]
            keep.append((bufs, pitches, chans))
            dests.append([(b.data_ptr(), p) for b, p in zip(bufs, pitches)])
        return dests, keep

    def timed(dec, streams, dests):
        batch, sources = dec.make_batch(streams, dests), dec.make_sources(addrs, lens)
        for _ in range(args.warmup + 2):
            st, _ = dec.parse_and_decode_batched(batch, sources, params)
            assert st == api.SUCCESS, st
        ts = []
        for _ in range(args.steps):
            for dv in range(torch.cuda.device_count()):
                torch.cuda.synchronize(dv)
            t0 = time.perf_counter()
            st, _ = dec.parse_and_decode_batched(batch, sources, params)
            ts.append(time.perf_counter() - t0)
            assert st == api.SUCCESS, st
        return 1e3 * sum(ts) / len(ts), dec.stats()

    streams = []
    for a, n in zip(addrs, lens):
        s = api.JpegStream()
        assert s.parse_ptr(a, n, arena) == api.SUCCESS
        streams.append(s)
    if single_ms is None:      # 1-GPU time of this workload through the same calls
        dec1 = api.Decoder(api.BACKEND_HARDWARE, dev0)
        dests0, keep0 = alloc([dev0] * len(datas))
        single_ms, _ = timed(dec1, streams, dests0)
        dec1.close()
    os.environ["ROCJPEG_B200_DEVICES"] = str(ndev)
    decn = api.Decoder(api.BACKEND_HARDWARE, dev0)
    del os.environ["ROCJPEG_B200_DEVICES"]
    used = decn.num_devices()
    out = {"devices_used": used, "single_gpu_ms": round(single_ms, 4)}
    orc = oracle.Oracle()
    ncount = torch.cuda.device_count()
    plan = api.plan_shards([s.info().raw_bytes for s in streams], used)
    for mode, devices in (("all_destinations_on_gpu0", [dev0] * len(datas)), ("destinations_colocated", [(dev0 + int(k)) % ncount for k in plan])):
        dests, keep = alloc(devices)
        ms, stn = timed(decn, streams, dests)
        ok = True
        for i in sorted(set([0, len(datas) // 3, len(datas) - 1])):   # a sample of the outputs against the oracle
            bufs, pitches, chans = keep[i]
            _, want = orc.decode(datas[i], fmt, pitches=pitches)
            for b, p, (rows, rb), wnt in zip(bufs, pitches, chans, want):
                got = b.cpu().numpy()[:rows * p].reshape(rows, p)[:, :rb]
                ok = ok and bool(np.array_equal(got, wnt[:rows, :rb]))
        out[mode] = {"ms_per_step": round(ms, 4), "value": round(total_px / 1e6 / (ms / 1e3), 1), "unit": UNIT,
                     "speedup_vs_1gpu": round(single_ms / ms, 3), "efficiency": round(single_ms / ms / used, 3),
                     "host_submit_ms": round(stn.host_submit_ms, 4), "host_wait_ms": round(stn.host_wait_ms, 4),
                     "devices": int(stn.devices), "verified_against_oracle": ok}
        del dests, keep
    decn.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOAD_DESC))
    ap.add_argument("--batch", type=int, default=0, help="override the number of images")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-budget", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--inlib-devices", type=int, default=0,
                    help="single process: also shard each rocJpegDecodeBatched call over this many GPUs inside the library "
                         "(ROCJPEG_B200_DEVICES); reported under `inlib` (under torchrun rank 0 does this with all N GPUs)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: every rank decodes a full batch; strong: one batch sharded over the ranks by scan bytes")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the pixels the last timed step decoded to DIR/image<i>_ch<c>.npy (float32, "
                         f"rank 0; where the whole batch would take more than {DUMP_BYTES >> 20} MiB, a seeded sample of rows, "
                         "whose indices go to image<i>_ch<c>_rows.npy)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the CUDA path decodes; the reference arm has no such outputs")
    if args.warmup < 3:
        sys.stderr.write(f"bench.py: --warmup {args.warmup} is below the 3 warm-up steps the timing rules require; using 3\n")
        args.warmup = 3
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    config = {"workload": f"{args.workload}: {WORKLOAD_DESC[args.workload]}", "per_gpu_batch": None,
              "output_format": None, "l2": "256 MiB device buffer written between timed steps (L2 flush)",
              "parallelism": f"{world} independent replicas, one process per GPU, no collective" if world > 1 else "single GPU"}

    if args.impl == "reference":
        # The reference cannot run without an AMD VCN engine and has no CPU path; the CPU arm is
        # the baseline BASELINE.json prescribes. Rank 0 alone runs it.
        if rank != 0:
            return
        datas, fmt = build_workload(args.workload, args.batch or None)
        config["per_gpu_batch"], config["output_format"] = len(datas), fmt
        per = max(2.0, min(args.cpu_budget, 60.0 / max(args.steps + args.warmup, 1)))
        for _ in range(min(args.warmup, 1)):
            run_cpu_baseline(datas, fmt, 0.5)
        t0 = time.perf_counter()
        mps, ips, threads, sample = run_cpu_baseline(datas, fmt, per * 3)
        line = {"impl": "reference", "metric": METRIC, "value": round(mps, 2), "unit": UNIT, "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(1e3 * len(datas) / ips, 3),
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/int32 (libjpeg-turbo islow)",
                "data": "synthetic", "config": config, "images_per_s": round(ips, 1),
                "cpu_baseline": {"value": round(mps, 2), "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                                 "host_cpus": os.cpu_count()},
                "e2e": {"value": round(mps, 2), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0, "wall_s": round(time.perf_counter() - t0, 2)}
        print(json.dumps(line))
        return

    import torch

    from rocjpeg_b200 import api

    assert torch.cuda.is_available(), "bench.py needs a CUDA device: rocjpeg_b200 has no CPU fallback"
    torch.cuda.set_device(local_rank)
    from rocjpeg_b200 import dist as rdist

    rdist.init("nccl", torch.device("cuda", local_rank))
    datas, fmt = build_workload(args.workload, args.batch or None)
    if args.scaling == "strong" and world > 1:
        mine = rdist.shard_by_cost([len(d) for d in datas], world)[rank]
        datas = [datas[i] for i in mine]
    total_px, dims = pixels_of(datas)
    config["per_gpu_batch"], config["output_format"] = len(datas), fmt
    config["scan_bytes_per_batch"] = sum(len(d) for d in datas)

    dec = api.Decoder(api.BACKEND_HARDWARE, local_rank)
    # The caller's JPEG files in page-locked host memory (one arena, every file at a 64-byte boundary): the
    # library reads them in place. rocJpegStreamParse walks the headers only; the entropy-coded bytes are first
    # touched by the upload inside rocJpegDecodeBatched and destuffed on the GPU.
    offs, total = [], 0
    for d in datas:
        offs.append(total)
        total += (len(d) + 63) // 64 * 64
    arena = torch.empty(total + 64, dtype=torch.uint8, pin_memory=True)
    arena_np = arena.numpy()
    for o, d in zip(offs, datas):
        arena_np[o:o + len(d)] = memoryview(d)
    addrs = [arena.data_ptr() + o for o in offs]
    lens = [len(d) for d in datas]
    streams = []
    t0 = time.perf_counter()
    for a, n in zip(addrs, lens):
        s = api.JpegStream()
        assert s.parse_ptr(a, n, arena) == api.SUCCESS
        streams.append(s)
    first_parse_s = time.perf_counter() - t0
    assert all(s.info().source_is_zero_copy for s in streams), "the pinned arena was not recognised as page-locked memory"
    dests, keep = [], []
    for (w, h, css) in dims:
        chans = api.output_channel_shapes(css, fmt, w, h)
        pitches = [rb for (_, rb) in chans]
        if fmt == "yuv_planar" and css in ("422", "420"):
            pitches[2] = pitches[1]
        bufs = [torch.empty(rows * p + 64, dtype=torch.uint8, device="cuda") for (rows, _), p in zip(chans, pitches)]
        keep.append((bufs, pitches, chans))
        dests.append([(b.data_ptr(), p) for b, p in zip(bufs, pitches)])
    params = api.make_params(fmt)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def l2_flush():
        flush.fill_(1)
        torch.cuda.synchronize()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            rdist.barrier()
            torch.cuda.synchronize()

    # ---- device-resident arm (value) -------------------------------------------------
    lanes_env = os.environ.get("ROCJPEG_B200_LANES")
    dec.set_profiling(2)   # first/last event only: the stages overlap as they do in production
    assert dec.prepare(streams, params, dests) == api.SUCCESS
    for _ in range(args.warmup):
        assert dec.run() == api.SUCCESS
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    step_ms, launches = [], 0
    wall0 = time.perf_counter()
    for _ in range(args.steps):
        l2_flush()
        assert dec.run() == api.SUCCESS
        st = dec.stats()
        step_ms.append(st.total_ms)
        launches += st.kernel_launches
    barrier()
    resident_wall = time.perf_counter() - wall0
    dumped = sample_outputs(torch, keep) if args.dump_outputs and rank == 0 else None
    resident_ms = sum(step_ms) / len(step_ms)
    stats = dec.stats()
    # per-stage device times for the roofline: the same resident batch on ONE pipeline lane, so that the
    # stages do not overlap each other (with several lanes the per-stage event times of the lanes add up)
    os.environ["ROCJPEG_B200_LANES"] = "1"
    dec.set_profiling(1)
    assert dec.prepare(streams, params, dests) == api.SUCCESS
    for _ in range(3):
        assert dec.run() == api.SUCCESS
    stage_ms, prof_steps, one_lane_ms = [0.0] * len(api.STAGES), max(3, min(args.steps, 10)), 0.0
    for _ in range(prof_steps):
        l2_flush()
        assert dec.run() == api.SUCCESS
        st = dec.stats()
        launches += st.kernel_launches
        one_lane_ms += st.total_ms
        for i in range(len(api.STAGES)):
            stage_ms[i] += st.stage_ms[i]
    stage_ms = [m / prof_steps for m in stage_ms]
    one_lane_ms /= prof_steps
    if lanes_env is None:
        del os.environ["ROCJPEG_B200_LANES"]
    else:
        os.environ["ROCJPEG_B200_LANES"] = lanes_env

    # ---- end-to-end arm (e2e): the public calls, raw JPEG files in host memory in -----------
    # Timed region = rocJpegStreamParse for every image + one rocJpegDecodeBatched (the caller's loop of the
    # reference's batched sample, issued from C: rocJpegB200ParseAndDecodeBatched), wall clock. Inside it: header
    # parse, host->device copy of the raw entropy-coded bytes and descriptors, GPU destuffing, decode, the
    # device->host read-back of the decoder's status words, stream sync.
    dec.set_profiling(False)                 # no stage events inside the timed call
    batch = dec.make_batch(streams, dests)   # the argument arrays a C caller holds ready
    sources = dec.make_sources(addrs, lens)
    for _ in range(args.warmup):
        st, _ = dec.parse_and_decode_batched(batch, sources, params)
        assert st == api.SUCCESS
    barrier()
    e2e_s, e2e_parse_s, e2e_launches = [], [], 0
    for _ in range(args.steps):
        l2_flush()
        t0 = time.perf_counter()
        rc, psec = dec.parse_and_decode_batched(batch, sources, params)
        e2e_s.append(time.perf_counter() - t0)
        e2e_parse_s.append(psec)
        assert rc == api.SUCCESS
        e2e_launches += dec.stats().kernel_launches
    barrier()
    e2e_stats = dec.stats()
    e2e_ms = 1e3 * sum(e2e_s) / len(e2e_s)
    parse_ms = 1e3 * sum(e2e_parse_s) / len(e2e_parse_s)
    # the same without the parse loop (the reference's samples leave parsing outside their timer)
    pre_s = []
    for _ in range(max(3, args.steps // 2)):
        l2_flush()
        t0 = time.perf_counter()
        rc = dec.decode_batched(batch, params)
        pre_s.append(time.perf_counter() - t0)
        assert rc == api.SUCCESS
    # ... and with the files in ordinary pageable memory (what the reference's samples hold them in): the parse
    # then copies the entropy-coded bytes into pooled page-locked staging
    pg_streams = []
    t0 = time.perf_counter()
    for d in datas:
        s = api.JpegStream()
        assert s.parse(d) == api.SUCCESS
        pg_streams.append(s)
    first_parse_pageable_s = time.perf_counter() - t0
    import ctypes as C

    pg_keep = [C.create_string_buffer(d, len(d)) for d in datas]
    pg_sources = dec.make_sources([C.addressof(b) for b in pg_keep], lens)
    pg_batch = dec.make_batch(pg_streams, dests)
    def pageable_pass():
        ts, ps = [], []
        for it in range(3 + max(3, args.steps // 2)):
            l2_flush()
            t0 = time.perf_counter()
            rc, psec = dec.parse_and_decode_batched(pg_batch, pg_sources, params)
            if it >= 3:
                ts.append(time.perf_counter() - t0)
                ps.append(psec)
            assert rc == api.SUCCESS
        return ts, ps

    pg_s, pg_parse_s = pageable_pass()
    os.environ["ROCJPEG_B200_DEFERRED_COPY"] = "1"      # opt-in: the decode call's helper threads copy, chunk by chunk
    pgd_s, pgd_parse_s = pageable_pass()
    del os.environ["ROCJPEG_B200_DEFERRED_COPY"]
    clocks = sampler.stop()
    dec.set_profiling(False)
    # ---- one call sharded inside the library over N GPUs (north star item 6, SURVEY.md section 8e) -----------------
    # Rank 0 alone, while the other ranks wait at a CPU barrier with idle GPUs: one rocJpegStreamParse x batch +
    # rocJpegDecodeBatched through a handle created with ROCJPEG_B200_DEVICES=N, (i) every destination on GPU 0
    # (the reference samples' layout: pixels of the peers' shares cross NVLink), (ii) destinations co-located with
    # the device the library's own plan gives each image (no pixel crosses a link).
    inlib = None
    ndev_inlib = world if world > 1 else args.inlib_devices
    if world > 1:
        rdist.cpu_barrier()
    if ndev_inlib > 1 and rank == 0 and torch.cuda.device_count() >= ndev_inlib:
        inlib = {"devices_requested": ndev_inlib, "single_gpu_e2e_ms": round(e2e_ms, 4), "workloads": {}}
        for wl in ([args.workload] if world == 1 else [args.workload, "c4_dri"]):
            inlib["workloads"][wl] = measure_inlib(api, torch, wl, args, ndev_inlib, local_rank,
                                                   (datas, fmt, dims, addrs, lens, arena, dests, e2e_ms) if wl == args.workload else None)
    if world > 1:
        rdist.cpu_barrier()

    # max over ranks
    pre_ms, pg_ms, pgd_ms = 1e3 * sum(pre_s) / len(pre_s), 1e3 * sum(pg_s) / len(pg_s), 1e3 * sum(pgd_s) / len(pgd_s)
    resident_ms, e2e_ms, pre_ms, pg_ms, pgd_ms = rdist.max_over_ranks([resident_ms, e2e_ms, pre_ms, pg_ms, pgd_ms], "cuda")
    px_all, n_all = rdist.sum_over_ranks([total_px, len(datas)], "cuda")
    if rank != 0:
        rdist.finalize()
        return

    mp_total = px_all / 1e6
    images_total = int(n_all)
    value = mp_total / (resident_ms / 1e3)
    peak, peak_src = measured_peaks()
    # Algorithmic bytes per stage, from what the stages actually move (SURVEY.md section 8d, DESIGN.md section 4):
    # entries = 32-bit coefficient entries K1 really wrote (counted on the device), 8-byte record per block.
    blocks, scan, entries = stats.blocks, stats.scan_bytes, stats.entries
    fused = stats.fused_blocks / blocks if blocks else 0.0      # share of the blocks the fused IDCT + output kernel handles
    k3_read = stats.plane_bytes * (1.0 - fused) if stage_ms[6] > 0 else 0
    coef_read = entries * 4 + blocks * 8                        # sparse entries + one record per block
    stage_bytes = {
        "destuff": scan * 2,                                    # raw bytes read, destuffed bytes written (re-read from L2 by the scatter pass)
        "huffman_sync": scan,                                   # count-only passes: the scan is read, a few words per subsequence written
        "huffman_write": scan + entries * 4 + blocks * 8,       # scan read; sparse entries + one record per block written
        "dc": blocks * 8 * 2,                                   # records read and rewritten
        "idct": (coef_read + blocks * 64) * (1.0 - fused),      # entries + records read, 64 samples per block written (un-fused pictures)
        "output": coef_read * fused + k3_read + stats.output_bytes,   # fused pictures: coefficients in, pixels out; others: planes read + pixels written
    }
    if stage_ms[3] <= 0.005:   # counting and write pass ran as one kernel (k1_fused): its time is under huffman_sync
        stage_bytes["huffman_sync"] = stage_bytes["huffman_write"]
    stages = {}
    for i, name in enumerate(api.STAGES):
        ms = stage_ms[i]
        b = stage_bytes.get(name)
        ran = ms > 0.005   # two back-to-back events are ~3 us apart: a stage below that launched nothing for this workload
        stages[name] = {"ms": round(ms, 4), "algorithmic_bytes": int(b) if b and ran else None,
                        "GB_s": round(b / ms / 1e6, 1) if b and ran else None,
                        "frac_of_hbm_peak": round(b / ms / 1e6 / peak, 4) if b and ran else None,
                        "traffic": measured_traffic(args.workload, name) if ran else None}
        if not ran and name != "upload":
            stages[name]["note"] = "no kernel of this stage runs for this workload"
    # dense-equivalent figure SURVEY.md section 8d quotes for the IDCT (128 B int16 block read + 64 B written)
    if stage_ms[5] > 0 and fused < 1.0:
        stages["idct"]["dense_equiv_GB_s"] = round(blocks * (1.0 - fused) * 192 / stage_ms[5] / 1e6, 1)
    if fused > 0:
        stages["output"]["note"] = f"{fused:.0%} of the blocks through the fused IDCT + output kernel (k23_fused: coefficient entries in, pixels out)"
    # `roofline`: the slower of the two HBM-bound stages the north star asks an HBM fraction for (IDCT, colour/output);
    # the entropy stage is latency/issue bound and reported as compressed GB/s + issue utilisation in `roofline_k1`
    hbm = [n for n in ("idct", "output") if stages[n]["ms"] > 0.005 and stage_bytes[n] > 0]
    dom = max(hbm, key=lambda n: stages[n]["ms"])
    dom_ms = stages[dom]["ms"]
    achieved = stage_bytes[dom] / dom_ms / 1e6 if dom_ms > 0 else 0.0
    k1_ms = stage_ms[2] + stage_ms[3]
    line = {
        "metric": METRIC, "value": round(value, 1), "unit": UNIT, "n_gpus": world, "steps": len(step_ms), "warmup": args.warmup,
        "ms_per_step": round(resident_ms, 4), "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "u8 / int16 coefficients / int32 IDCT / fp32 colour", "data": "synthetic", "config": config,
        "images_per_s": round(images_total / (resident_ms / 1e3), 1),
        "value_note": "device-resident: raw entropy-coded bytes + descriptors already in HBM (rocJpegB200Prepare); each step = "
                      "rocJpegB200Run = every kernel of the path (destuff, Huffman, DC, IDCT, output), CUDA events",
        "e2e": {"value": round(mp_total / (e2e_ms / 1e3), 1), "unit": UNIT, "images_per_s": round(images_total / (e2e_ms / 1e3), 1),
                "ms_per_step": round(e2e_ms, 4), "h2d_bytes_per_step": int(e2e_stats.h2d_bytes), "d2h_bytes_per_step": int(e2e_stats.d2h_bytes),
                "parse_ms_per_batch": round(parse_ms, 4), "first_parse_ms": round(first_parse_s * 1e3, 3),
                "note": "rocJpegStreamParse x batch + rocJpegDecodeBatched, wall clock, starting from the caller's raw JPEG files in "
                        "page-locked host memory (read in place); pixels left in device memory as the API specifies"},
        "e2e_preparsed": {"value": round(mp_total / (pre_ms / 1e3), 1), "unit": UNIT, "ms_per_step": round(pre_ms, 4),
                          "note": "rocJpegDecodeBatched alone on already parsed streams (what the reference's samples time)"},
        "e2e_pageable": {"value": round(mp_total / (pg_ms / 1e3), 1), "unit": UNIT, "ms_per_step": round(pg_ms, 4),
                         "parse_ms_per_batch": round(1e3 * sum(pg_parse_s) / len(pg_parse_s), 4),
                         "first_parse_ms": round(first_parse_pageable_s * 1e3, 3),
                         "note": "same as e2e with the files in pageable memory (what the reference's samples hold them in): the parse copies "
                                 "the entropy-coded bytes into pooled page-locked staging on the caller's thread",
                         "deferred_copy": {"value": round(mp_total / (pgd_ms / 1e3), 1), "ms_per_step": round(pgd_ms, 4),
                                           "parse_ms_per_batch": round(1e3 * sum(pgd_parse_s) / len(pgd_parse_s), 4),
                                           "note": "ROCJPEG_B200_DEFERRED_COPY=1: the decode call's helper threads copy, chunk by chunk "
                                                   "ahead of each chunk's upload"}},
        "gpu_launches": int(launches + e2e_launches),
        "launches_per_step": int(stats.kernel_launches),
        "roofline": {"bound": "hbm", "kernel": dom, "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                     "frac": round(achieved / peak, 4), "traffic": measured_traffic(args.workload, dom), "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": int(stage_bytes[dom]), "launch_ms": dom_ms,
                     "issue_utilisation": (measured_traffic(args.workload, "issue") or {}).get("k2_idct" if dom == "idct" else "k23_warp"),
                     "note": "slower of the two stages the north star names HBM-bound (IDCT, output); both are in fact bound by issue slots "
                             "(issue_utilisation: committed ncu capture); every stage's own fraction is in `stages`"},
        "roofline_k1": {"bound": "latency/issue", "compressed_GB_s": round(scan / (k1_ms or 1e-9) / 1e6, 2), "ms": round(k1_ms, 4),
                        "sync_ms": round(stage_ms[2], 4), "write_ms": round(stage_ms[3], 4),
                        "entries_written_GB_s": round((entries * 4 + blocks * 8) / ((stage_ms[3] if stage_ms[3] > 0.005 else k1_ms) or 1e-9) / 1e6, 1),
                        "fused": stage_ms[3] <= 0.005,
                        "issue_utilisation": measured_traffic(args.workload, "k1_issue"),
                        "note": "entropy stage: compressed bitstream GB/s over k1_sync + k1_write (fused: one kernel, k1_fused, its time under "
                                "sync_ms; entries_written_GB_s then over the whole kernel); issue-slot utilisation from the committed "
                                "ncu capture (profiles/)"},
        "stages": stages, "stages_note": "CUDA-event time per stage of the same resident batch on one pipeline lane "
                                         f"(stages serialised; that step takes {round(one_lane_ms, 4)} ms)",
        "k1": {"lanes": stats.lanes, "subsequence_bytes": stats.subsequence_bytes, "subsequences": int(stats.subsequences), "sync_rounds": stats.sync_rounds,
               "decodes_per_round": [int(x) for x in stats.decodes_per_round[:stats.sync_rounds]], "entries": int(entries)},
        "clocks": clocks, "resident_wall_s": round(resident_wall, 3),
        "e2e_host": {"submit_ms": round(e2e_stats.host_submit_ms, 4), "wait_ms": round(e2e_stats.host_wait_ms, 4)},
    }
    if inlib:
        line["inlib"] = inlib
    if not args.no_cpu_baseline:
        mps, ips, threads, sample = run_cpu_baseline(datas, fmt, args.cpu_budget)
        line["cpu_baseline"] = {"value": round(mps, 2), "unit": UNIT, "images_per_s": round(ips, 1), "cores": threads, "kind": "port",
                                "sample": sample, "host_cpus": os.cpu_count()}
    if dumped is not None:
        write_outputs(args.dump_outputs, dumped)
    print(json.dumps(line))
    rdist.finalize()


if __name__ == "__main__":
    main()

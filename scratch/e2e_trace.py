"""Timeline of one end-to-end call (ROCJPEG_B200_TRACE=2) plus wall-clock e2e over a few settings.

  python scratch/e2e_trace.py [workload] [steps]
Run under gpurun; each configuration runs in a child process (the knobs are read once per process).
"""
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def child(workload, steps):
    import torch

    from rocjpeg_b200 import api, datagen

    datas, fmt = datagen.workload(workload, None)
    dec = api.Decoder(api.BACKEND_HARDWARE, 0)
    offs, total = [], 0
    for d in datas:
        offs.append(total)
        total += (len(d) + 63) // 64 * 64
    arena = torch.empty(total + 64, dtype=torch.uint8, pin_memory=True)
    an = arena.numpy()
    for o, d in zip(offs, datas):
        an[o:o + len(d)] = memoryview(d)
    addrs = [arena.data_ptr() + o for o in offs]
    lens = [len(d) for d in datas]
    streams, dims = [], []
    for a, n in zip(addrs, lens):
        s = api.JpegStream()
        assert s.parse_ptr(a, n, arena) == api.SUCCESS
        i = s.info()
        dims.append((i.width, i.height, api.CSS_NAME[i.chroma_subsampling]))
        streams.append(s)
    dests, keep = [], []
    for (w, h, css) in dims:
        chans = api.output_channel_shapes(css, fmt, w, h)
        pitches = [rb for (_, rb) in chans]
        if fmt == "yuv_planar" and css in ("422", "420"):
            pitches[2] = pitches[1]
        bufs = [torch.empty(rows * p + 64, dtype=torch.uint8, device="cuda") for (rows, _), p in zip(chans, pitches)]
        keep.append(bufs)
        dests.append([(b.data_ptr(), p) for b, p in zip(bufs, pitches)])
    params = api.make_params(fmt)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    batch = dec.make_batch(streams, dests)
    sources = dec.make_sources(addrs, lens)
    quiet = os.environ.get("ROCJPEG_B200_TRACE", "0") == "0"
    for _ in range(5):
        st, _ = dec.parse_and_decode_batched(batch, sources, params)
        assert st == api.SUCCESS
    ts = []
    for _ in range(steps):
        flush.fill_(1)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        rc, psec = dec.parse_and_decode_batched(batch, sources, params)
        ts.append(time.perf_counter() - t0)
        assert rc == api.SUCCESS
    ts.sort()
    st = dec.stats()
    px = sum(w * h for (w, h, _) in dims)
    # resident: Prepare once, Run per step, first-to-last event
    dec.set_profiling(2)
    assert dec.prepare(streams, params, dests) == api.SUCCESS
    for _ in range(5):
        assert dec.run() == api.SUCCESS
    rs = []
    for _ in range(steps):
        flush.fill_(1)
        torch.cuda.synchronize()
        assert dec.run() == api.SUCCESS
        rs.append(dec.stats().total_ms)
    rs.sort()
    print(f"RESIDENT {os.environ.get('CFG_NAME')}: mean {sum(rs) / len(rs):.4f} ms, median {rs[len(rs) // 2]:.4f}, min {rs[0]:.4f}", flush=True)
    print(f"RESULT {os.environ.get('CFG_NAME')}: e2e mean {1e3 * sum(ts) / len(ts):.4f} ms, median {1e3 * ts[len(ts) // 2]:.4f}, min {1e3 * ts[0]:.4f} "
          f"({px / 1e6 / (sum(ts) / len(ts)) / 1e3:.1f} GMP/s) submit {st.host_submit_ms:.3f} wait {st.host_wait_ms:.3f} lanes {st.lanes}", flush=True)


def main():
    workload = sys.argv[1] if len(sys.argv) > 1 else "c3"
    steps = int(sys.argv[2]) if len(sys.argv) > 2 else 20
    if os.environ.get("CFG_NAME"):
        return child(workload, steps)
    configs = [
        ("default+trace", {"ROCJPEG_B200_TRACE": "2"}, 3),
        ("default", {}, steps),
        ("lanes1", {"ROCJPEG_B200_LANES": "1"}, steps),
        ("lanes2", {"ROCJPEG_B200_LANES": "2"}, steps),
        ("lanes3", {"ROCJPEG_B200_LANES": "3"}, steps),
        ("lanes4_equal", {"ROCJPEG_B200_LANES": "4", "ROCJPEG_B200_SPLIT": "25,25,25,25"}, steps),
        ("lanes4_40_30_20_10", {"ROCJPEG_B200_LANES": "4", "ROCJPEG_B200_SPLIT": "40,30,20,10"}, steps),
        ("nomerge", {"ROCJPEG_B200_NO_MERGE": "1"}, steps),
        ("lanes4_15_30_30_25", {"ROCJPEG_B200_LANES": "4", "ROCJPEG_B200_SPLIT": "15,30,30,25"}, steps),
        ("lanes4_20_35_30_15", {"ROCJPEG_B200_LANES": "4", "ROCJPEG_B200_SPLIT": "20,35,30,15"}, steps),
        ("s64", {"ROCJPEG_B200_SUBSEQ": "64"}, steps),
        ("halo4", {"ROCJPEG_B200_HALO": "4"}, steps),
        ("halo8", {"ROCJPEG_B200_HALO": "8"}, steps),
        ("nok1fuse", {"ROCJPEG_B200_NO_K1_FUSE": "1"}, steps),
        ("lanes5", {"ROCJPEG_B200_LANES": "5"}, steps),
        ("lanes6", {"ROCJPEG_B200_LANES": "6"}, steps),
    ]
    for sp in filter(None, os.environ.get("E2E_SPLITS", "").split(";")):
        configs.append(("split_" + sp.replace(",", "_"), {"ROCJPEG_B200_LANES": str(len(sp.split(","))), "ROCJPEG_B200_SPLIT": sp}, steps))
    extra = os.environ.get("E2E_CONFIGS")
    for name, env, n in configs:
        if extra and name not in extra.split(",") and not name.startswith("split_"):
            continue
        e = dict(os.environ)
        e.update(env)
        e["CFG_NAME"] = name
        r = subprocess.run([sys.executable, os.path.abspath(__file__), workload, str(n)], env=e, capture_output=True, text=True, timeout=300)
        out = (r.stdout + r.stderr).splitlines()
        if name.endswith("trace"):
            keep = [l for l in out if l.startswith("[rocjpeg_b200]") or l.startswith("RES")]
            print("\n".join(keep[-(3 * 6 + 1):]), flush=True)
        else:
            print("\n".join(l for l in out if l.startswith("RESULT") or l.startswith("RESIDENT") or "Error" in l or "error" in l), flush=True)


if __name__ == "__main__":
    main()

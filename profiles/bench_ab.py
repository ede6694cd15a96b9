"""A/B of two builds of librocjpeg.so under bench.py: the builds alternate run by run (ROCJPEG_B200_LIB selects one),
the first run of each on a workload also writes --dump-outputs, and those files are compared byte for byte. Prints one
JSON line per run, a header line with the card's name, power limit and maximum SM clock, and one line per workload
saying whether the outputs are identical.

    python profiles/bench_ab.py --parent LIB --new LIB [--workloads c2,c3,c5_400] [--runs 5] [--steps 50] [--warmup 10]
"""
import argparse
import filecmp
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i", "0"],
                       capture_output=True, text=True)
    name, power, mhz = [x.strip() for x in r.stdout.strip().split(",")]
    return {"gpu": name, "power_limit_w": float(power), "sm_max_mhz": float(mhz)}


def run(lib, workload, steps, warmup, dump):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", str(warmup),
           "--workload", workload, "--no-cpu-baseline"] + (["--dump-outputs", dump] if dump else [])
    r = subprocess.run(cmd, capture_output=True, text=True, env={**os.environ, "ROCJPEG_B200_LIB": lib}, cwd=ROOT)
    if r.returncode != 0:
        sys.exit(f"bench.py failed ({lib}, {workload}):\n{r.stdout}\n{r.stderr}")
    return json.loads(r.stdout.strip().splitlines()[-1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent", required=True)
    ap.add_argument("--new", required=True)
    ap.add_argument("--workloads", default="c2,c3,c5_400")
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    args = ap.parse_args()
    print(json.dumps({**card(), "what": f"bench.py --gpus 1 --steps {args.steps} --warmup {args.warmup} --no-cpu-baseline; parent "
                      f"build and this build alternated, {args.runs} runs each, one GPU call; --dump-outputs of the first run of each "
                      "compared byte for byte"}), flush=True)
    builds = {"parent": os.path.abspath(args.parent), "new": os.path.abspath(args.new)}
    with tempfile.TemporaryDirectory() as tmp:
        for w in args.workloads.split(","):
            dumps = {b: os.path.join(tmp, f"{w}_{b}") for b in builds}
            for i in range(args.runs):
                for b in (("parent", "new") if i % 2 == 0 else ("new", "parent")):
                    line = run(builds[b], w, args.steps, args.warmup, dumps[b] if i == 0 else None)
                    print(json.dumps({"workload": w, "build": b, "ms_per_step": line["ms_per_step"], "e2e_ms": line["e2e"]["ms_per_step"],
                                      "launches_per_step": line["launches_per_step"], "e2e_host": line["e2e_host"],
                                      "clocks": line["clocks"]}), flush=True)
            names = sorted(os.listdir(dumps["parent"]))
            same = names == sorted(os.listdir(dumps["new"])) and all(
                filecmp.cmp(os.path.join(dumps["parent"], n), os.path.join(dumps["new"], n), shallow=False) for n in names)
            print(json.dumps({"workload": w, "outputs_identical": same, "files": len(names)}), flush=True)


if __name__ == "__main__":
    main()

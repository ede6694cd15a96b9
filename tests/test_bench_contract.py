"""bench.py contract checks: the reference arm (the CPU baseline BASELINE.json prescribes) prints one JSON line with the
keys a caller reads, without a GPU; on the GPU, --dump-outputs writes what the timed steps decoded."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--batch", "6", "--steps", "1",
                        "--warmup", "3", "--cpu-budget", "0.3"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    j = json.loads(lines[0])
    assert j["impl"] == "reference" and j["unit"] == "MP/s" and j["higher_is_better"] is True
    assert j["metric"] == "decoded_MP_per_s_rocJpegDecodeBatched" and j["value"] > 0
    assert j["config"]["workload"].startswith("c3") and j["config"]["per_gpu_batch"] == 6
    assert j["cpu_baseline"]["kind"] in ("port", "reference") and j["cpu_baseline"]["cores"] >= 1
    assert j["cpu_baseline"]["value"] == j["value"]
    assert j["e2e"] == {"value": j["value"], "unit": "MP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


@pytest.mark.gpu
def test_dumped_outputs_are_what_the_timed_steps_decoded(tmp_path):
    """--dump-outputs on a batch too large to dump whole: per channel of every picture, the seeded sample of rows
    (float32) and their indices, equal to the oracle's decode of the same seeded input at those rows; the line reports
    the number of timed steps that ran."""
    import numpy as np

    import oracle
    from rocjpeg_b200 import datagen

    n = 32   # 32 x 500 x 375 x 3 float32 samples: above the dump budget, so rows are sampled
    out = tmp_path / "outputs"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--batch", str(n), "--steps", "7", "--warmup", "3",
                        "--no-cpu-baseline", "--dump-outputs", str(out)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr
    j = json.loads([l for l in r.stdout.splitlines() if l.strip()][-1])
    assert j["steps"] == 7
    names = [f"image{i:04d}_ch{c}" for i in range(n) for c in range(3)]
    assert sorted(p.name for p in out.iterdir()) == sorted([m + ".npy" for m in names] + [m + "_rows.npy" for m in names])
    assert sum(p.stat().st_size for p in out.iterdir()) < 64e6
    datas, fmt = datagen.workload("c3", n)
    orc = oracle.Oracle()
    kept = 0
    for i, d in enumerate(datas):
        info, want = orc.decode(d, fmt)
        for c, ((rows, rb), w) in enumerate(zip(oracle.output_shapes(info, fmt), want)):
            got = np.load(out / f"image{i:04d}_ch{c}.npy")
            idx = np.load(out / f"image{i:04d}_ch{c}_rows.npy")
            assert got.dtype == np.float32 and idx.dtype == np.float32
            idx = idx.astype(np.int64)
            assert len(idx) < rows and np.all(np.diff(idx) > 0) and idx[-1] < rows
            assert np.array_equal(got, w[idx, :rb].astype(np.float32)), (i, c)
            kept += len(idx)
    assert kept > 0


def test_reference_arm_is_silent_on_other_ranks():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--batch", "6", "--gpus", "2"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""

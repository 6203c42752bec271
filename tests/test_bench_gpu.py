"""bench.py on the GPU: --steps is the number of timed steps, and --dump-outputs writes the detections block of the last one,
bit-identical to the oracle on the input set that step reads (the inputs depend on the arguments only)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
from fdt_b200 import synth
from oracle import oracle as orc

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_is_the_last_timed_step(tmp_path):
    steps, warmup = 5, 3                                   # the last step reads input set 1: an off-by-one in the count shows
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", str(warmup),
                        "--no-secondary", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                       cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps and line["timing"]["steps"] == steps
    assert line["gpu_launches"] == line["gpu_launches_per_step"] * steps
    assert sorted(os.listdir(tmp_path)) == ["detections.npy"]
    got = np.load(tmp_path / "detections.npy")
    assert got.dtype == np.float32 and got.shape == (bench.B_PER_GPU, 2, bench.TOP_K, 5)
    # steps are numbered from 0 over warm-up and timed steps alike; step i reads input set i % ROTATE
    last = max(warmup, 3) + steps - 1
    pri = synth.priors_numpy(bench.WIDTH, bench.HEIGHT)
    loc, conf = synth.detect_inputs(bench.B_PER_GPU, pri, bench.SEED + 1000 * (last % bench.ROTATE), bench.CONF_T, "random")
    want = orc.Detect(2, 0, bench.TOP_K, bench.CONF_T, bench.NMS_T)(loc, conf, pri)
    assert np.array_equal(got.view(np.int32), want.view(np.int32))

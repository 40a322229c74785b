"""bench.py end to end at two timed steps: the JSON line reports the steps asked for, and --dump-outputs writes the
reconstruction the timed (graph-replayed) step returned."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from util import rel_l2

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_times_the_asked_steps_and_dumps_the_reconstruction(tmp_path):
    run = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "0", "--no-cpu",
                          "--no-extras", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900)
    assert run.returncode == 0, run.stderr[-3000:]
    line = json.loads(run.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2 and line["value"] > 0
    assert os.listdir(tmp_path) == ["reconstruction.npy"]
    rec = np.load(tmp_path / "reconstruction.npy")
    assert rec.dtype == np.float32 and rec.shape == (16, 1, 256, 256) and np.isfinite(rec).all()

    import bench
    dev = torch.device("cuda:0")
    with torch.random.fork_rng(devices=[0]):        # build_model seeds the global generators
        radon, model = bench.build_model(dev)
    sparse = bench.synthetic_sparse_sinograms(radon, dev, bench.BATCH, seed=100)
    with torch.no_grad():
        want = model(sparse)
    # the benchmark autotunes cuDNN (TF32 convolutions): another algorithm may round differently
    assert rel_l2(torch.from_numpy(rec), want) < 1e-2

"""bench.py --dump-outputs: the arrays written after the timed steps are what a caller of the timed path receives
for bench.py's own seeded inputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import restatement as R

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench_dump(out_dir, workload):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", workload, "--steps", "2",
                          "--warmup", "1", "--no-cpu", "--dump-outputs", str(out_dir)],
                         capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-3000:]
    assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == 2
    return {f[:-len(".npy")]: np.load(os.path.join(out_dir, f)) for f in os.listdir(out_dir)}


def test_dump_of_the_rcca_fit(tmp_path):
    import bench
    from cca_zoo_b200.linear import rCCA

    got = _bench_dump(tmp_path, "rcca")
    assert sorted(got) == ["means_0", "means_1", "weights_0", "weights_1"]
    bench.W.update(bench.WORKLOADS["rcca"])
    est = rCCA(latent_dimensions=64, c=0.1, precision="tf32x3b").fit(
        [torch.from_numpy(v).cuda() for v in bench.make_views(1000)])
    for i in range(2):
        assert got[f"weights_{i}"].dtype == est.weights_[i].dtype and got[f"weights_{i}"].shape == (1024, 64)
        np.testing.assert_allclose(got[f"means_{i}"], est.means_[i], rtol=1e-5, atol=1e-6)
    assert R.max_rel_err_per_vector([got["weights_0"].astype(np.float64), got["weights_1"].astype(np.float64)],
                                    [w.astype(np.float64) for w in est.weights_]) < 1e-3


def test_dump_of_the_ccaloss_step(tmp_path):
    import bench
    from cca_zoo_b200.deep import CCALoss

    got = _bench_dump(tmp_path, "ccaloss64")
    assert sorted(got) == ["grad_0", "grad_1", "loss"]
    bench.W.update(bench.WORKLOADS["ccaloss64"])
    zs = [z.cuda().requires_grad_(True) for z in bench.make_representations(0)]
    loss = CCALoss(eps=1e-5)(zs)
    loss.backward()
    assert got["loss"].dtype == np.float32 and abs(float(got["loss"]) - loss.item()) < 1e-4 * abs(loss.item())
    for i, z in enumerate(zs):
        g = z.grad.cpu().numpy()
        assert got[f"grad_{i}"].shape == (4096, 64)
        assert np.abs(got[f"grad_{i}"] - g).max() < 1e-3 * np.abs(g).max()

"""World-size-2 run of the sharded LM on two GPUs (NCCL plumbing + NVLink peer-memory data path): the trajectories must
reproduce the reference's single-process goldens (tests/golden/lm.npz).  Needs two CUDA devices."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.mark.gpu
def test_sharded_lm_two_gpus_matches_reference(tmp_path, golden_lm):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    out = str(tmp_path / "nccl.npz")
    port = str(_free_port())
    procs = []
    for rank in range(2):
        env = dict(os.environ, RANK=str(rank), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT=port, PYTHONPATH=ROOT)
        procs.append(subprocess.Popen([sys.executable, os.path.join(ROOT, "tests", "nccl_worker.py"), out], env=env,
                                      stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    logs = [p.communicate(timeout=900)[0] for p in procs]
    assert all(p.returncode == 0 for p in procs), "\n".join(logs)
    r, g = np.load(out), golden_lm
    assert r["peer_available"][0] == 1 and r["poseinv_peer"][0] == 1 and r["reproj_peer"][0] == 1, "NVLink peer route not taken"
    np.testing.assert_allclose(r["poseinv_loss"], g["poseinv/trustregion/loss"], rtol=1e-5, atol=1e-20)
    np.testing.assert_allclose(r["poseinv_poses"], g["poseinv/trustregion/poses"][-1], atol=1e-9)
    for case in ("reproj", "reproj_hard"):
        for tag in (case, case + "_gather", case + "_sorted", case + "_gather_sorted"):   # exchange forms x row splits
            assert r[f"{tag}_peer"][0] == 1
            np.testing.assert_allclose(r[f"{tag}_loss"], g[f"{case}/trustregion/loss"], rtol=1e-6)
            np.testing.assert_allclose(r[f"{tag}_poses"], g[f"{case}/trustregion/poses"][-1], atol=1e-8)
            np.testing.assert_array_equal(r[f"{tag}_reject"], g[f"{case}/trustregion/reject"])
    np.testing.assert_allclose(r["pgo_loss"], g["pgo/trustregion/loss"], rtol=1e-6)
    np.testing.assert_allclose(r["pgo_poses"], g["pgo/trustregion/poses"][-1], atol=1e-7)
    np.testing.assert_allclose(r["ba_loss"], g["ba/trustregion/loss"], rtol=1e-5)
    np.testing.assert_allclose(r["ba_poses"], g["ba/trustregion/poses"][-1], atol=1e-6)
    np.testing.assert_allclose(r["ba_points"], g["ba/trustregion/points"][-1], atol=1e-6)

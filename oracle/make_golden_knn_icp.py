"""Record knn, ReduceToBason and ICP results of the REFERENCE (pypose v0.9.5, fp64, CPU) for tests/golden/knn_icp.npz:

    python oracle/make_golden_knn_icp.py

TEST INFRASTRUCTURE ONLY.  Cases:
  * `knn` (pypose/function/geometry.py:228-313) on seeded clouds: several shapes, D, ord and k, largest on and off,
    broadcast batches, and clouds with duplicated points (ties);
  * `ReduceToBason` (pypose/utils/stepper.py): the step / stop sequence and the verbose text for scalar and batched
    loss sequences, including a reset between two runs;
  * `ICP` (pypose/module/icp.py): the geometry of the reference's `test_icp_batch` (an L-shaped wall and a noisy arc,
    two transforms) and both broadcasting patterns on a synthetic cloud (the reference's laser scans need a download).
"""
import contextlib
import io
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.environ.get("PYPOSE_REFERENCE", "/root/reference"))
sys.dont_write_bytecode = True
import pypose as ref  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests", "golden", "knn_icp.npz")
ORD = {1: 1, 2: 2, float("inf"): 0}


def knn_cases(g, rng):
    def cloud(*shape):
        return torch.from_numpy(rng.standard_normal(shape))

    dup = cloud(40, 3)
    dup = torch.cat([dup, dup[:13], dup[5:9]], 0)[torch.from_numpy(rng.permutation(57))]
    grid = torch.from_numpy(np.stack(np.meshgrid(*[np.arange(4.0)] * 3, indexing="ij"), -1).reshape(-1, 3))
    cases = [
        ("small", cloud(6, 3), cloud(4, 3), 2, 2, False),
        ("d3_l2", cloud(33, 3), cloud(300, 3), 8, 2, False),
        ("d3_l1", cloud(33, 3), cloud(300, 3), 5, 1, False),
        ("d3_inf", cloud(33, 3), cloud(300, 3), 3, float("inf"), False),
        ("d3_far", cloud(31, 3), cloud(257, 3), 8, 2, True),
        ("d1", cloud(17, 1), cloud(70, 1), 4, 2, False),
        ("d5_k32", cloud(9, 5), cloud(100, 5), 32, 2, False),
        ("d8_inf_far", cloud(9, 8), cloud(64, 8), 7, float("inf"), True),
        ("batch", cloud(2, 20, 3), cloud(2, 90, 3), 4, 2, False),
        ("bcast_ref", cloud(20, 3), cloud(3, 90, 3), 2, 1, False),
        ("bcast_nbr", cloud(2, 1, 20, 3), cloud(3, 90, 3), 3, 2, False),
        ("dup", dup, dup, 4, 2, False),
        ("dup_far", dup[:20], dup, 6, 1, True),
        ("grid", grid[:30], grid, 8, 2, False),
    ]
    for name, r, n, k, o, largest in cases:
        v, i = ref.knn(r, n, k=k, ord=o, largest=largest)
        g[f"knn/{name}/ref"], g[f"knn/{name}/nbr"] = r.numpy(), n.numpy()
        g[f"knn/{name}/values"], g[f"knn/{name}/indices"] = v.numpy(), i.numpy()
        g[f"knn/{name}/args"] = np.array([k, ORD[o], int(largest)])


def stepper_cases(g):
    seqs = {
        "scalar": ([0.81, 0.6561, 0.43, 0.1853, 0.0343, 0.0012, 0.0012, 0.0012], dict(steps=20, patience=2, decreasing=0.1)),
        "plateau": ([1.0, 0.9999, 0.9998, 0.9998, 0.9997, 0.9997, 0.9996], dict(steps=50)),
        "tol": ([1.0, 1e-3, 1e-6, 1e-7], dict(steps=10)),
        "maxsteps": ([1.0, 0.5, 0.25, 0.125, 0.0625], dict(steps=3)),
        "batched": ([[1.0, 2.0], [0.5, 1.99999], [0.25, 1.99998], [0.2499, 1.99997], [0.2498, 1.99996], [1e-6, 1e-6]],
                    dict(steps=30, patience=2)),
    }
    for name, (losses, kw) in seqs.items():
        st = ref.utils.ReduceToBason(verbose=True, **kw)
        rows, text = [], io.StringIO()
        for run in range(2):                   # a second run after reset(): patience_count carries over
            st.reset()
            with contextlib.redirect_stdout(text):
                for loss in losses:
                    if not st.continual():
                        break
                    st.step(torch.tensor(loss, dtype=torch.float64))
                    rows.append([run, st.steps, int(st.continual()), st.patience_count])
        g[f"stepper/{name}/losses"] = np.array(losses, dtype=np.float64)
        g[f"stepper/{name}/kwargs"] = np.array([kw.get("steps"), kw.get("patience", 5), kw.get("decreasing", 1e-3),
                                                kw.get("tol", 1e-5)], dtype=np.float64)
        g[f"stepper/{name}/trace"] = np.array(rows, dtype=np.int64)
        g[f"stepper/{name}/text"] = np.array(text.getvalue())


def icp_batch_geometry():
    """reference tests/module/test_icp.py::test_icp_batch, seeded."""
    torch.manual_seed(0)
    n = 1000
    x1, y1, z1 = torch.linspace(0, 10, n // 2), torch.zeros(n // 2), torch.zeros(n // 2)
    x2, y2, z2 = torch.full((n // 2,), 10.0), torch.linspace(20, 0, n // 2), torch.zeros(n // 2)
    wall = torch.stack((torch.cat((x1, x2)), torch.cat((y1, y2)), torch.cat((z1, z2))), dim=1)
    theta = torch.linspace(0, 0.5 * 3.14159265, n)
    arc = torch.stack((10 + 10 * torch.cos(theta) + torch.randn(n), 20 - 10 * torch.sin(theta) + torch.randn(n),
                       torch.randn(n)), dim=1)
    source = torch.stack((wall, arc), dim=0).double()
    tf = ref.SE3(torch.tensor([[-5.05, -3.02, 0.02, 0, 0, 0.0499792, 0.9987503],
                               [-2, 1, 1, 0.1304815, 0.0034168, -0.025953, 0.9911051]], dtype=torch.float64))
    return source, tf.unsqueeze(-2).Act(source), tf


def synthetic_cloud(rng, n=600):
    """A scan-like cloud: points on three walls, a floor patch and a ball, with a little noise."""
    u = rng.uniform(0, 1, size=(n, 2))
    part = rng.integers(0, 4, size=n)
    p = np.where(part[:, None] == 0, np.stack([u[:, 0] * 8, np.zeros(n), u[:, 1] * 2], 1),
        np.where(part[:, None] == 1, np.stack([np.full(n, 8.0), u[:, 0] * 5, u[:, 1] * 2], 1),
        np.where(part[:, None] == 2, np.stack([np.zeros(n), u[:, 0] * 5, u[:, 1] * 2], 1),
                 np.stack([u[:, 0] * 8, u[:, 1] * 5, np.zeros(n)], 1))))
    ball = rng.standard_normal((n // 4, 3))
    ball = 0.8 * ball / np.linalg.norm(ball, axis=1, keepdims=True) + np.array([5.0, 3.0, 1.0])
    return torch.from_numpy(np.concatenate([p, ball]) + 0.01 * rng.standard_normal((n + n // 4, 3)))


def icp_cases(g, rng):
    source, target, tf = icp_batch_geometry()
    g["icp/batch/source"], g["icp/batch/target"], g["icp/batch/tf"] = source.numpy(), target.numpy(), tf.tensor().numpy()
    g["icp/batch/result"] = ref.module.ICP()(source, target).tensor().numpy()

    pc1 = synthetic_cloud(rng)
    pc2 = pc1 + 0.005 * torch.from_numpy(rng.standard_normal(pc1.shape))
    tf1 = ref.SE3(torch.tensor([[-0.05, -0.02, 0.0, 0, 0, 0.0499792, 0.9987503]] * 2, dtype=torch.float64))
    tgt = tf1.unsqueeze(-2).Act(pc2)
    g["icp/bcast1/source"], g["icp/bcast1/target"] = pc1.numpy(), tgt.numpy()
    g["icp/bcast1/result"] = ref.module.ICP()(pc1, tgt).tensor().numpy()

    tf2 = ref.SE3(torch.tensor([[-0.05, -0.02, 0.0, 0, 0, 0.0499792, 0.9987503],
                                [-0.01, -0.03, 0.0, 0, 0, 0.0499792, 0.9987503]], dtype=torch.float64))
    src = tf2.unsqueeze(-2).Act(pc1)
    stepper = ref.utils.ReduceToBason(steps=100, patience=3)
    g["icp/bcast2/source"], g["icp/bcast2/target"] = src.numpy(), pc2.numpy()
    g["icp/bcast2/result"] = ref.module.ICP(stepper=stepper)(src, pc2).tensor().numpy()

    init = ref.SE3(torch.tensor([0.1, 0.0, 0.0, 0, 0, 0, 1], dtype=torch.float64))
    g["icp/init/init"] = init.tensor().numpy()
    g["icp/init/result"] = ref.module.ICP(init=init)(pc1, tgt[0]).tensor().numpy()
    g["icp/l1/result"] = ref.module.ICP()(pc1, tgt[0], ord=1).tensor().numpy()


def main():
    rng = np.random.default_rng(2026)
    g = {}
    knn_cases(g, rng)
    stepper_cases(g)
    icp_cases(g, rng)
    np.savez_compressed(OUT, **g)
    print("wrote", OUT, len(g), "arrays")


if __name__ == "__main__":
    main()

"""pp.knn and pp.module.ICP on the B200 (csrc/knn.cu): against the reference's recorded results
(tests/golden/knn_icp.npz) and against a chunked fp64 brute force on the device, on both sides of the N2 split."""
import math
import os

import numpy as np
import pytest
import torch

import pypose_b200 as pp
from pypose_b200.function import _knn

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = torch.device("cuda:0")


@pytest.fixture(scope="module")
def golden_knn_icp():
    return np.load(os.path.join(ROOT, "tests", "golden", "knn_icp.npz"))


def brute(ref, nbr, k, ord, largest, chunk=2048):
    """fp64 distances of the k (+1, for tie detection) best neighbours, ties by the lower index (stable sort)."""
    r, n = ref.double(), nbr.double()
    vals, idx = [], []
    kk = min(k + 1, n.shape[-2])
    for i in range(0, r.shape[-2], chunk):
        d = torch.cdist(r[..., i:i + chunk, :], n, p=ord, compute_mode="donot_use_mm_for_euclid_dist")
        s, j = torch.sort(d, dim=-1, descending=largest, stable=True)
        vals.append(s[..., :kk])
        idx.append(j[..., :kk])
    return torch.cat(vals, -2), torch.cat(idx, -2)


def check(ref, nbr, k, ord, largest, v, i, tol):
    bv, bi = brute(ref, nbr, k, ord, largest)
    ev = bv[..., :k]
    assert torch.allclose(v.double(), ev, rtol=tol, atol=tol), (v.double() - ev).abs().max().item()
    # indices are exact wherever the oracle has no tie within the tolerance
    gap = (bv[..., 1:] - bv[..., :-1]).abs() <= tol * (1 + bv[..., 1:].abs())
    tie = torch.zeros_like(ev, dtype=torch.bool)
    tie[..., 1:] |= gap[..., :k - 1]
    m = min(k, gap.shape[-1])
    tie[..., :m] |= gap[..., :m]
    assert (i[~tie] == bi[..., :k][~tie]).all()
    # every returned index is at the returned distance
    nb = nbr.double().expand(*i.shape[:-2], *nbr.shape[-2:])
    pts = torch.gather(nb, -2, i.reshape(*i.shape[:-2], -1, 1).expand(*i.shape[:-2], i.shape[-2] * k, nbr.shape[-1]))
    d = torch.linalg.vector_norm(ref.double().unsqueeze(-2) - pts.reshape(*i.shape, -1), ord=ord, dim=-1)
    assert torch.allclose(d, ev, rtol=tol, atol=tol)


TOL = {torch.float32: 1e-6, torch.float64: 1e-12}


def test_knn_matches_golden(golden_knn_icp):
    g = golden_knn_icp
    names = sorted({key.split("/")[1] for key in g.files if key.startswith("knn/")})
    for dtype in (torch.float64, torch.float32):
        for name in names:
            k, code, largest = (int(x) for x in g[f"knn/{name}/args"])
            o = {0: math.inf, 1: 1, 2: 2}[code]
            r = torch.from_numpy(g[f"knn/{name}/ref"]).to(DEV, dtype)
            n = torch.from_numpy(g[f"knn/{name}/nbr"]).to(DEV, dtype)
            v, i = pp.knn(r, n, k=k, ord=o, largest=bool(largest))
            ev = torch.from_numpy(g[f"knn/{name}/values"]).to(DEV)
            tol = TOL[dtype]
            assert torch.allclose(v.double(), ev, rtol=tol, atol=tol), (name, dtype)
            check(r, n, k, o, bool(largest), v, i, tol)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("ord", [1, 2, math.inf])
@pytest.mark.parametrize("N", [1, 31, 33, 255, 256, 257, 1000])
def test_knn_sizes_ords_against_brute_force(dtype, ord, N):
    g = torch.Generator(device=DEV).manual_seed(N)
    ref = torch.randn(N, 3, device=DEV, dtype=dtype, generator=g)
    nbr = torch.randn(max(N, 40), 3, device=DEV, dtype=dtype, generator=g)
    for k in (1, 8, 32):
        k = min(k, nbr.shape[0])
        for largest in (False, True):
            v, i = pp.knn(ref, nbr, k=k, ord=ord, largest=largest)
            check(ref, nbr, k, ord, largest, v, i, TOL[dtype])


@pytest.mark.parametrize("D", [1, 2, 4, 5, 8])
def test_knn_point_dimensions(D):
    ref = torch.randn(2, 300, D, device=DEV, dtype=torch.float64)
    nbr = torch.randn(2, 700, D, device=DEV, dtype=torch.float64)
    v, i = pp.knn(ref, nbr, k=5)
    check(ref, nbr, 5, 2, False, v, i, 1e-12)


def test_knn_large_2_17():
    N = 1 << 17
    g = torch.Generator(device=DEV).manual_seed(17)
    ref = torch.rand(N, 3, device=DEV, generator=g)
    nbr = torch.rand(N, 3, device=DEV, generator=g)
    sel = torch.randperm(N, device=DEV, generator=g)[:4096]
    for k in (1, 8):
        v, i = pp.knn(ref, nbr, k=k)
        check(ref[sel], nbr, k, 2, False, v[sel], i[sel], 1e-6)


def test_knn_duplicates_follow_the_tie_rule():
    g = torch.Generator(device=DEV).manual_seed(5)
    base = torch.randint(0, 4, (200, 3), device=DEV, generator=g).double()      # a 4x4x4 lattice: many equal distances
    for dtype in (torch.float32, torch.float64):
        x = base.to(dtype)
        for largest in (False, True):
            for o in (1, 2, math.inf):
                v, i = pp.knn(x, x, k=32, ord=o, largest=largest)
                eq = v[:, 1:] == v[:, :-1]
                assert (i[:, 1:][eq] > i[:, :-1][eq]).all()
                _, bi = brute(x, x, 32, o, largest)
                assert torch.equal(i, bi[:, :32])
        first = torch.stack([torch.nonzero((base == p).all(-1))[0, 0] for p in base])
        assert torch.equal(pp.knn(x, x, k=1).indices[:, 0], first)


def test_knn_nan_orders_above_finite():
    ref = torch.zeros(1, 3, device=DEV)
    nbr = torch.tensor([[1.0, 0, 0], [float("nan"), 0, 0], [2.0, 0, 0]], device=DEV)
    v, i = pp.knn(ref, nbr, k=3)
    assert i.tolist() == [[0, 2, 1]] and torch.isnan(v[0, 2])
    v, i = pp.knn(ref, nbr, k=3, largest=True)
    assert i.tolist() == [[1, 2, 0]] and torch.isnan(v[0, 0])


def test_knn_non_contiguous_and_broadcast_inputs():
    big = torch.randn(3, 500, 6, device=DEV, dtype=torch.float64)
    ref = big[:, ::2, 1:4]                        # strided view
    nbr = torch.randn(3, 3, 400, device=DEV, dtype=torch.float64).transpose(-1, -2)
    assert not ref.is_contiguous() and not nbr.is_contiguous()
    v, i = pp.knn(ref, nbr, k=4)
    check(ref, nbr, 4, 2, False, v, i, 1e-12)
    one = torch.randn(300, 3, device=DEV, dtype=torch.float64)
    v, i = pp.knn(one, nbr, k=4)                  # one query cloud for every batch: passed once, stride 0
    check(one.expand(3, 300, 3), nbr, 4, 2, False, v, i, 1e-12)
    v, i = pp.knn(ref.unsqueeze(0), nbr.unsqueeze(1), k=2, ord=1)
    assert v.shape == (3, 3, 250, 2)
    check(ref.unsqueeze(0).expand(3, 3, 250, 3), nbr.unsqueeze(1).expand(3, 3, 400, 3), 2, 1, False, v, i, 1e-12)


@pytest.mark.parametrize("N1,N2,k,split", [(64, 60000, 8, True), (2000, 2000, 1, True), (1 << 19, 1000, 1, False),
                                           (4096, 100000, 32, True), (200000, 5000, 32, False)])
def test_knn_both_sides_of_the_split(N1, N2, k, split):
    ref = torch.randn(N1, 3, device=DEV)
    nbr = torch.randn(N2, 3, device=DEV)
    S, _ = _knn._plan(1, N1, N2, k, ref)
    assert (S > 1) == split
    v, i = pp.knn(ref, nbr, k=k)
    sel = torch.arange(0, N1, max(1, N1 // 2048), device=DEV)
    check(ref[sel], nbr, k, 2, False, v[sel], i[sel], 1e-6)


@pytest.mark.parametrize("k", [1, 16])
def test_knn_memory_is_linear_in_queries(k):
    N = 100000
    ref = torch.rand(N, 3, device=DEV)
    nbr = torch.rand(N, 3, device=DEV)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.max_memory_allocated()
    v, i = pp.knn(ref, nbr, k=k)
    torch.cuda.synchronize()
    grown = torch.cuda.max_memory_allocated() - base
    assert grown < 64 * 2 ** 20, grown          # the reference's difference tensor would be 120 GB


@pytest.mark.parametrize("ord", [1, 2, math.inf])
def test_knn_gradcheck(ord):
    g = torch.Generator(device=DEV).manual_seed(3)
    ref = torch.randn(2, 7, 3, device=DEV, dtype=torch.float64, generator=g).requires_grad_()
    nbr = torch.randn(40, 3, device=DEV, dtype=torch.float64, generator=g).requires_grad_()
    assert torch.autograd.gradcheck(lambda r, n: pp.knn(r, n, k=4, ord=ord).values, (ref, nbr))
    assert torch.autograd.gradcheck(lambda r, n: pp.knn(r, n, k=3, ord=ord, largest=True).values, (ref, nbr))


def posediff(ref, est):
    T = ref * est.Inv()
    dt = torch.linalg.norm(T.translation(), dim=-1)
    dr = 2 * torch.acos(T.tensor()[..., 6].abs().clamp(max=1))
    return dt.mean().item(), dr.mean().item()


@pytest.mark.parametrize("dtype,tol", [(torch.float64, 1e-5), (torch.float32, 1e-3)])
@pytest.mark.parametrize("case", ["batch", "bcast1", "bcast2", "init", "l1"])
def test_icp_matches_golden(golden_knn_icp, dtype, tol, case):
    g = golden_knn_icp
    src_key = {"init": "bcast1", "l1": "bcast1"}.get(case, case)
    source = torch.from_numpy(g[f"icp/{src_key}/source"]).to(DEV, dtype)
    target = torch.from_numpy(g[f"icp/{src_key}/target"]).to(DEV, dtype)
    stepper = pp.utils.ReduceToBason(steps=100, patience=3) if case == "bcast2" else None
    init, extra = None, {}
    if case in ("init", "l1"):
        target = target[0]
    if case == "init":
        init = pp.SE3(torch.from_numpy(g["icp/init/init"]).to(DEV, dtype))
    if case == "l1":
        extra["ord"] = 1
    result = pp.module.ICP(init=init, stepper=stepper)(source, target, **extra)
    expect = torch.from_numpy(g[f"icp/{case}/result"]).to(DEV, dtype)
    assert result.shape == expect.shape and result.dtype == dtype
    dt, dr = posediff(pp.SE3(expect), result)
    assert dt < tol and dr < tol, (dt, dr)


def test_icp_batch_geometry_meets_the_reference_test(golden_knn_icp):
    g = golden_knn_icp
    source = torch.from_numpy(g["icp/batch/source"]).to(DEV, torch.float32)
    tf = pp.SE3(torch.from_numpy(g["icp/batch/tf"]).to(DEV, torch.float32))
    target = tf.unsqueeze(-2).Act(source)
    dt, dr = posediff(tf, pp.module.ICP()(source, target))
    assert dt < 0.1 and dr < 0.1


@pytest.mark.parametrize("dtype,tol_t", [(torch.float64, 1e-6), (torch.float32, 5e-2)])
def test_icp_far_from_origin_converges(dtype, tol_t):
    """1e5 points offset by +1e3 in every axis: the centred cross-covariance comes from fp64 raw moments.  In fp32 the
    points themselves are quantised to 6e-5 there and the estimate to about 1e-2 in translation."""
    g = torch.Generator(device=DEV).manual_seed(11)
    n = 100000
    cloud = (torch.rand(n, 3, device=DEV, generator=g, dtype=torch.float64)
             * torch.tensor([10.0, 10.0, 2.0], device=DEV, dtype=torch.float64) + 1e3)
    q = torch.tensor([0.0, 0.0, 0.0043633, 0.9999905], device=DEV, dtype=torch.float64)
    tf = pp.SE3(torch.cat([torch.tensor([0.03, -0.02, 0.01], device=DEV, dtype=torch.float64), q / q.norm()]))
    target = tf.Act(cloud - 1e3) + 1e3                            # a small motion about a corner of the cloud
    o = torch.full((3,), 1e3, device=DEV, dtype=torch.float64)
    truth = pp.SE3(torch.cat([tf.translation() + o - tf.rotation().Act(o), tf.tensor()[3:]]))
    result = pp.module.ICP()(cloud.to(dtype), target.to(dtype))
    dt, dr = posediff(truth, pp.SE3(result.tensor().double()))
    assert dt < tol_t and dr < 1e-3, (dt, dr)

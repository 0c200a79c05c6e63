"""pp.knn, pp.utils.ReduceToBason and pp.module.ICP without a GPU: the API (shapes, broadcasting, the named-tuple
return, the ValueErrors at each limit), the stepper against the reference's recorded step sequences, the knn backward,
and the ICP control flow against the reference's transforms (tests/golden/knn_icp.npz, oracle/make_golden_knn_icp.py).

The package registers CUDA kernels only; the fixture below gives `b200pose::knn` and `b200pose::icp_moments` test-only
CPU implementations backed by a numpy brute force, for the duration of this module."""
import contextlib
import io
import math
import os

import numpy as np
import pytest
import torch

import pypose_b200 as pp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def brute_knn(ref, nbr, k, code, largest):
    """numpy: (..., N1, D), (..., N2, D) -> values, indices (..., N1, k); ties by the lower index."""
    r, n = ref.detach().double().numpy(), nbr.detach().double().numpy()
    diff = r[..., :, None, :] - n[..., None, :, :]
    d = (np.sqrt((diff ** 2).sum(-1)) if code == 2 else np.abs(diff).sum(-1) if code == 1
         else np.abs(diff).max(-1))
    idx = np.argsort(-d if largest else d, axis=-1, kind="stable")[..., :k]
    return d, idx


def brute_moments(source, target, pose, code):
    """numpy ICP moments for (batch, 7) poses, matching csrc/knn.cu: count, sum s', sum t, sum t s'^T, sum dist."""
    from oracle import lie_oracle as O
    batch = tuple(pose.shape[:-1])
    s = np.broadcast_to(source.detach().double().numpy(), batch + tuple(source.shape[-2:]))
    t = np.broadcast_to(target.detach().double().numpy(), batch + tuple(target.shape[-2:]))
    P = np.broadcast_to(pose.detach().double().numpy()[..., None, :], s.shape[:-1] + (7,))
    sp = O.run("SE3_act_fwd", np.ascontiguousarray(P.reshape(-1, 7)), np.ascontiguousarray(s.reshape(-1, 3)))[0]
    sp = sp.reshape(s.shape).copy()
    d, idx = brute_knn(torch.from_numpy(sp), torch.from_numpy(np.ascontiguousarray(t)), 1, code, False)
    idx = idx[..., 0]
    dist = np.take_along_axis(d, idx[..., None], -1)[..., 0]
    tn = np.take_along_axis(t, idx[..., None], -2)
    m = np.concatenate([np.full(batch + (1,), s.shape[-2], dtype=np.float64), sp.sum(-2), tn.sum(-2),
                        np.einsum("...na,...nb->...ab", tn, sp).reshape(batch + (9,)), dist.sum(-1)[..., None]], -1)
    return torch.from_numpy(m)


@pytest.fixture(scope="module", autouse=True)
def cpu_kernels():
    lib = torch.library.Library("b200pose", "IMPL")

    def knn_cpu(ref, nbr, k, code, largest):
        d, idx = brute_knn(ref, nbr, k, code, largest)
        v = np.take_along_axis(d, idx, -1)
        return torch.from_numpy(v).to(ref.dtype), torch.from_numpy(idx).long()

    lib.impl("knn", knn_cpu, "CPU")
    lib.impl("icp_moments", brute_moments, "CPU")
    yield
    lib._destroy()


@pytest.fixture(scope="module")
def golden_knn_icp():
    return np.load(os.path.join(ROOT, "tests", "golden", "knn_icp.npz"))


def test_knn_returns_topk_named_tuple_with_reference_example():
    ref = torch.tensor([[9., 2., 2.], [1., 0., 2.], [0., 1., 1.], [5., 0., 1.], [1., 0., 1.], [5., 5., 3.]])
    nbr = torch.tensor([[1., 0., 1.], [1., 6., 2.], [5., 1., 0.], [9., 0., 2.]])
    out = pp.knn(ref, nbr, k=2)
    assert isinstance(out, torch.return_types.topk)
    assert out.indices.dtype == torch.int64 and out.values.shape == (6, 2)
    assert out.indices.tolist() == [[3, 2], [0, 2], [0, 2], [2, 0], [0, 2], [1, 2]]
    assert torch.allclose(out.values[:, 0], torch.tensor([2.0, 1.0, 2 ** 0.5, 2 ** 0.5, 0.0, 18 ** 0.5]))


@pytest.mark.parametrize("rs,ns,expect", [
    ((7, 3), (2, 9, 3), (2, 7, 4)),
    ((2, 7, 3), (9, 3), (2, 7, 4)),
    ((2, 1, 7, 3), (3, 9, 3), (2, 3, 7, 4)),
    ((1, 7, 3), (4, 9, 3), (4, 7, 4)),
])
def test_knn_broadcasts_batch_dimensions(rs, ns, expect):
    ref, nbr = torch.randn(rs, dtype=torch.float64), torch.randn(ns, dtype=torch.float64)
    v, i = pp.knn(ref, nbr, k=4)
    assert v.shape == expect and i.shape == expect
    full = torch.broadcast_shapes(ref.shape[:-2], nbr.shape[:-2])
    d, idx = brute_knn(ref.expand(*full, *rs[-2:]), nbr.expand(*full, *ns[-2:]), 4, 2, False)
    assert np.array_equal(i.numpy(), idx)


@pytest.mark.parametrize("kwargs,match", [
    (dict(k=0), "k must be"), (dict(k=33), "k must be"), (dict(k=10), "k must be"),
    (dict(ord=3), "ord must be"), (dict(ord="fro"), "ord must be"), (dict(dim=0), "last dimension"),
])
def test_knn_limits_raise_value_error(kwargs, match):
    with pytest.raises(ValueError, match=match):
        pp.knn(torch.randn(5, 3), torch.randn(9, 3), **kwargs)


def test_knn_shape_and_dtype_limits_raise_value_error():
    with pytest.raises(ValueError, match="D must be"):
        pp.knn(torch.randn(5, 9), torch.randn(9, 9))
    with pytest.raises(ValueError, match="D must be"):
        pp.knn(torch.randn(5, 0), torch.randn(9, 0))
    with pytest.raises(ValueError, match="same point dimension"):
        pp.knn(torch.randn(5, 3), torch.randn(9, 2))
    with pytest.raises(ValueError, match="float32"):
        pp.knn(torch.randn(5, 3).half(), torch.randn(9, 3).half())
    with pytest.raises(ValueError, match="float32"):
        pp.knn(torch.randn(5, 3), torch.randn(9, 3, dtype=torch.float64))
    with pytest.raises(ValueError, match="broadcast"):
        pp.knn(torch.randn(2, 5, 3), torch.randn(3, 9, 3))
    with pytest.raises(ValueError, match="shape"):
        pp.knn(torch.randn(3), torch.randn(9, 3))
    v, i = pp.knn(torch.randn(5, 8), torch.randn(32, 8), k=32, dim=1)     # the limits themselves are accepted
    assert v.shape == (5, 32)


def test_knn_sorted_false_still_sorted_and_largest_descends():
    ref, nbr = torch.randn(6, 3, dtype=torch.float64), torch.randn(40, 3, dtype=torch.float64)
    v = pp.knn(ref, nbr, k=7, sorted=False).values
    assert (v[:, 1:] >= v[:, :-1]).all()
    v = pp.knn(ref, nbr, k=7, largest=True).values
    assert (v[:, 1:] <= v[:, :-1]).all()


def test_knn_matches_golden_through_the_wrapper(golden_knn_icp):
    g = golden_knn_icp
    names = sorted({key.split("/")[1] for key in g.files if key.startswith("knn/")})
    assert len(names) >= 10
    for name in names:
        k, code, largest = (int(x) for x in g[f"knn/{name}/args"])
        o = {0: math.inf, 1: 1, 2: 2}[code]
        v, i = pp.knn(torch.from_numpy(g[f"knn/{name}/ref"]), torch.from_numpy(g[f"knn/{name}/nbr"]), k=k, ord=o,
                      largest=bool(largest))
        np.testing.assert_allclose(v.numpy(), g[f"knn/{name}/values"], rtol=1e-12, atol=1e-12, err_msg=name)


@pytest.mark.parametrize("ord", [1, 2, math.inf])
def test_knn_backward_gradcheck(ord):
    torch.manual_seed(0)
    ref = torch.randn(2, 6, 3, dtype=torch.float64, requires_grad=True)
    nbr = torch.randn(15, 3, dtype=torch.float64, requires_grad=True)
    assert torch.autograd.gradcheck(lambda r, n: pp.knn(r, n, k=3, ord=ord).values, (ref, nbr))
    assert torch.autograd.gradcheck(lambda r, n: pp.knn(r, n, k=2, ord=ord, largest=True).values, (ref, nbr))


def test_knn_backward_is_zero_at_zero_distance():
    x = torch.randn(5, 3, dtype=torch.float64, requires_grad=True)
    for o in (1, 2, math.inf):
        v = pp.knn(x, x.detach(), k=1, ord=o).values
        assert (v == 0).all()
        g, = torch.autograd.grad(v.sum(), x)
        assert (g == 0).all()


@pytest.mark.parametrize("name", ["scalar", "plateau", "tol", "maxsteps", "batched"])
def test_reduce_to_bason_matches_golden_sequences(golden_knn_icp, name):
    g = golden_knn_icp
    steps, patience, decreasing, tol = g[f"stepper/{name}/kwargs"]
    st = pp.utils.ReduceToBason(int(steps), patience=int(patience), decreasing=decreasing, tol=tol, verbose=True)
    rows, text = [], io.StringIO()
    for run in range(2):
        st.reset()
        with contextlib.redirect_stdout(text):
            for loss in g[f"stepper/{name}/losses"]:
                if not st.continual():
                    break
                st.step(torch.tensor(loss, dtype=torch.float64))
                rows.append([run, st.steps, int(st.continual()), st.patience_count])
    assert np.array_equal(np.array(rows), g[f"stepper/{name}/trace"])
    assert text.getvalue() == str(g[f"stepper/{name}/text"])


def test_reduce_to_bason_accepts_python_floats():
    st = pp.utils.ReduceToBason(steps=5, patience=2, decreasing=0.1)
    x = 0.9
    n = 0
    while st.continual():
        x = x ** 2
        st.step(x)
        n += 1
    assert n == 5 and st.steps == 5


@pytest.mark.parametrize("case,kw", [("batch", {}), ("bcast1", {}), ("bcast2", {"patience": 3, "steps": 100}),
                                     ("init", {}), ("l1", {})])
def test_icp_matches_golden_transforms(golden_knn_icp, case, kw):
    g = golden_knn_icp
    src_key = {"init": "bcast1", "l1": "bcast1"}.get(case, case)
    source = torch.from_numpy(g[f"icp/{src_key}/source"])
    target = torch.from_numpy(g[f"icp/{src_key}/target"])
    stepper = pp.utils.ReduceToBason(**kw) if kw else None
    init, extra = None, {}
    if case in ("init", "l1"):
        target = target[0]
    if case == "init":
        init = pp.SE3(torch.from_numpy(g["icp/init/init"]))
    if case == "l1":
        extra["ord"] = 1
    result = pp.module.ICP(init=init, stepper=stepper)(source, target, **extra)
    expect = g[f"icp/{case}/result"]
    assert pp.is_SE3(result) and tuple(result.shape) == expect.shape
    q, qe = result.tensor()[..., 3:].numpy(), expect[..., 3:]
    q = q * np.sign((q * qe).sum(-1, keepdims=True))            # q and -q are the same rotation
    np.testing.assert_allclose(result.tensor()[..., :3].numpy(), expect[..., :3], atol=1e-5)
    np.testing.assert_allclose(q, qe, atol=1e-5)


def test_icp_rejects_unsupported_arguments():
    icp = pp.module.ICP()
    with pytest.raises(ValueError, match="ord"):
        icp(torch.randn(5, 3), torch.randn(6, 3), ord=3)
    with pytest.raises(ValueError, match="last dimension"):
        icp(torch.randn(5, 3), torch.randn(6, 3), dim=0)
    with pytest.raises(ValueError, match="shape"):
        icp(torch.randn(5, 2), torch.randn(6, 2))


def test_operands_on_different_devices_raise_value_error():
    cpu, meta = torch.randn(5, 3), torch.randn(9, 3, device="meta")
    with pytest.raises(ValueError, match="same device"):
        pp.knn(cpu, meta)
    with pytest.raises(ValueError, match="same device"):
        pp.module.ICP()(cpu, meta)


def test_icp_rejects_a_non_se3_initial_transform():
    with pytest.raises(ValueError, match="SE3"):
        pp.module.ICP(init=pp.randn_SO3())
    with pytest.raises(ValueError, match="SE3"):
        pp.module.ICP()(torch.randn(5, 3), torch.randn(6, 3), init=torch.zeros(7))

"""Lie launches that read what the launch before them is still writing, back to back on one stream (no synchronize
in between), as the streaming shell's programmatic dependent launch lets them overlap.  Each check replays the same
launches one at a time with a device synchronize after each, and requires bit-identical results.
"""
import ctypes

import pytest
import torch

from pypose_b200 import _C

pytestmark = pytest.mark.gpu
SFX = {torch.float32: "f32", torch.float64: "f64"}
# 1e6: the bench's batch; 1 / 3: tail kernel only; 257 / 4099: TMA body + <= 3-row tail; 25600 = 100 tiles of
# 256 rows, fewer than the grid's CTA slots on any current GPU
SIZES = [1_000_000, 1, 3, 257, 4099, 25600]


def call(sym, ins, outs, n, stream):
    rc = _C.fn(sym)(*[ctypes.c_void_p(t.data_ptr()) for t in ins + outs], n, ctypes.c_void_p(stream.cuda_stream))
    assert rc == 0, (sym, rc)


def chain(x, X, dtype, stream):
    """Exp -> Log -> Exp -> Log on the same two buffers: every launch reads the previous launch's output, and every
    launch but the first two overwrites a buffer that the launch before the previous one read."""
    s = SFX[dtype]
    n = x.shape[0]
    return [(f"b200_se3_exp_fwd_{s}", [x], [X], n), (f"b200_SE3_log_fwd_{s}", [X], [x], n),
            (f"b200_se3_exp_fwd_{s}", [x], [X], n), (f"b200_SE3_log_fwd_{s}", [X], [x], n)]


def one_at_a_time(launches, stream):
    for sym, ins, outs, n in launches:
        call(sym, ins, outs, n, stream)
        torch.cuda.synchronize()


def back_to_back(launches, stream, graph):
    if not graph:
        for sym, ins, outs, n in launches:
            call(sym, ins, outs, n, stream)
        torch.cuda.synchronize()
        return
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=stream):
        for sym, ins, outs, n in launches:
            call(sym, ins, outs, n, torch.cuda.current_stream())
    g.replay()
    torch.cuda.synchronize()


def se3_inputs(n, dtype, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randn(n, 6, dtype=dtype, device="cuda", generator=g) * 0.8


@pytest.mark.parametrize("graph", [False, True], ids=["eager", "graph"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("n", SIZES)
def test_exp_log_chain_back_to_back(n, dtype, graph):
    x0 = se3_inputs(n, dtype, n)
    ref_x, ref_X = x0.clone(), torch.empty(n, 7, dtype=dtype, device="cuda")
    x, X = x0.clone(), torch.empty(n, 7, dtype=dtype, device="cuda")
    side = torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        one_at_a_time(chain(ref_x, ref_X, dtype, side), side)
        back_to_back(chain(x, X, dtype, side), side, graph)
    assert torch.equal(X, ref_X)
    assert torch.equal(x, ref_x)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["f32", "f64"])
def test_lie_launch_after_torch_kernel(dtype):
    """The torch kernel that writes Exp's input never triggers its dependents: Exp still has to see all its writes."""
    n = 1_000_000
    src = se3_inputs(n, dtype, 7)
    x, X = torch.empty_like(src), torch.empty(n, 7, dtype=dtype, device="cuda")
    ref_X = torch.empty_like(X)
    side = torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        call(f"b200_se3_exp_fwd_{SFX[dtype]}", [src * 0.5], [ref_X], n, side)
        torch.cuda.synchronize()
        x.fill_(float("nan"))                  # stale values Exp must never pick up
        torch.cuda.synchronize()
        torch.mul(src, 0.5, out=x)
        call(f"b200_se3_exp_fwd_{SFX[dtype]}", [x], [X], n, side)
        torch.cuda.synchronize()
    assert torch.equal(X, ref_X)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("n", [1_000_000, 4099])
def test_two_input_op_on_previous_output(n, dtype):
    """SE3_mul reads the group element Exp is still writing, and a second operand nobody writes."""
    s = SFX[dtype]
    x, z = se3_inputs(n, dtype, 11), se3_inputs(n, dtype, 12)
    Z = torch.empty(n, 7, dtype=dtype, device="cuda")
    side = torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        call(f"b200_se3_exp_fwd_{s}", [z], [Z], n, side)
        torch.cuda.synchronize()
        outs = []
        for run in (one_at_a_time, lambda l, st: back_to_back(l, st, False)):
            X, W = torch.empty(n, 7, dtype=dtype, device="cuda"), torch.empty(n, 7, dtype=dtype, device="cuda")
            run([(f"b200_se3_exp_fwd_{s}", [x], [X], n), (f"b200_SE3_mul_fwd_{s}", [X, Z], [W], n)], side)
            outs.append(W)
    assert torch.equal(outs[0], outs[1])

"""DEV ONLY: time the candidate shells of libvariants.so (variants.cu) on the bench's sequence.
Per candidate: Exp alone and Log alone (CUDA graph over a ring of 8 batches, each launch its own buffers) and the
Exp j -> Log j step (the bench's 8-step graph).  N = AB_N (1e6); both dtypes of every candidate in the library.
usage: python tools/variants/ab.py [name-prefix ...]     env: B200POSE_PDL, B200POSE_CTAS_PER_SM"""
import ctypes, json, os, re, sys
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "libvariants.so")
lib = ctypes.CDLL(LIB)
N = int(os.environ.get("AB_N", 1_000_000))
src = open(os.path.join(HERE, "variants.cu")).read()
cands = ["%s_s%so%s_pf%s" % m for m in re.findall(r"^PAIR\(\w+, (f\d\d), (\d+), (\d+), (\d+)\)", src, re.M)]
if sys.argv[1:]:
    cands = [c for c in cands if any(c.startswith(a) for a in sys.argv[1:])]
ring, dev = 8, torch.device("cuda")


def fn(name, ct):
    f = getattr(lib, name)
    f.restype = ctypes.c_int
    f.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_longlong, ctypes.c_void_p]
    return f


def timed(seq, reps):
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        seq(ctypes.c_void_p(side.cuda_stream))
        side.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            seq(ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    for _ in range(3):
        g.replay()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        g.replay()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e3 / (reps * ring)


bufs = {}
for dt in (torch.float32, torch.float64):
    gen = torch.Generator(device=dev).manual_seed(0)
    xs = [torch.randn(N, 6, device=dev, dtype=dt, generator=gen) * 0.5 for _ in range(ring)]
    bufs[dt] = (xs, [torch.empty(N, 7, device=dev, dtype=dt) for _ in range(ring)],
                [torch.empty(N, 6, device=dev, dtype=dt) for _ in range(ring)])
res = {}
for rnd in range(2):                       # two rounds, candidates interleaved: the spread is visible per candidate
    for c in cands:
        dt = torch.float32 if c.startswith("f32") else torch.float64
        xs, Xs, ys = bufs[dt]
        fe, fl = fn("exp_" + c, dt), fn("log_" + c, dt)
        pe = lambda sp: [fe(xs[j].data_ptr(), Xs[j].data_ptr(), N, sp) for j in range(ring)]
        pl = lambda sp: [fl(Xs[j].data_ptr(), ys[j].data_ptr(), N, sp) for j in range(ring)]
        ps = lambda sp: [(fe(xs[j].data_ptr(), Xs[j].data_ptr(), N, sp), fl(Xs[j].data_ptr(), ys[j].data_ptr(), N, sp))
                         for j in range(ring)]
        r = res.setdefault(c, {"exp": [], "log": [], "step": []})
        r["exp"].append(round(timed(pe, 200), 2))
        r["log"].append(round(timed(pl, 200), 2))
        r["step"].append(round(timed(ps, 200), 2))
print(json.dumps({"pdl": os.environ.get("B200POSE_PDL", "1"), "ctas": os.environ.get("B200POSE_CTAS_PER_SM", "max"),
                  "n": N, "gpu": torch.cuda.get_device_name(), "us": res}))

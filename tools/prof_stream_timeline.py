"""Dev tool: per-CTA timeline of the streaming shell across launch boundaries, in the bench's own sequence.

usage: python tools/prof_stream_timeline.py [--lib tools/variants/libtrace.so] [--out FILE.json]

Drives the trace build of the shell (tools/variants/trace.cu, built by tools/variants/build.sh) with the bench's
headline sequence: se3 Exp j, SE3 Log j, Exp j+1, ... over a ring of 8 (x, X, y) batches at N = 1e6 fp32, captured
in one CUDA graph of 16 launches.  The graph is replayed twice back to back and every CTA's %globaltimer stamps are
read back: entry, after griddepcontrol.wait, tile 0 landed, last store issued, exit.

Per launch it prints
  span   first CTA entry -> last CTA exit
  gap    previous launch's last exit -> this launch's first tile landed (the boundary cost the read pipeline pays)
  rel    previous launch's last exit -> first CTA past griddepcontrol.wait
  ovl    per SM, time CTAs of this and the previous launch are resident together (mean over SMs)
The timer's resolution is measured first; stamps coarser than ~0.5 us cannot resolve the gaps, and the tool says so.
"""
import argparse
import ctypes
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def timer_resolution(lib, dev):
    n = 8192
    buf = torch.empty(n, dtype=torch.int64, device=dev)
    assert lib.trace_timer_samples(ctypes.c_void_p(buf.data_ptr()), n, None) == 0
    torch.cuda.synchronize()
    d = np.diff(buf.cpu().numpy())
    nz = d[d > 0]
    return {"min_step_ns": int(nz.min()) if nz.size else None, "median_step_ns": float(np.median(nz)) if nz.size else None,
            "ticks": int(nz.size), "reads": n}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", default=os.path.join(ROOT, "tools", "variants", "libtrace.so"))
    ap.add_argument("--out", default=None)
    ap.add_argument("--n", type=int, default=1_000_000)
    args = ap.parse_args()
    lib = ctypes.CDLL(args.lib)
    for f in (lib.trace_se3_exp_fwd_f32, lib.trace_SE3_log_fwd_f32):
        f.restype = ctypes.c_int
        f.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_longlong, ctypes.c_void_p]
    lib.trace_read.restype = ctypes.c_longlong
    lib.trace_capacity.restype = ctypes.c_longlong
    lib.trace_timer_samples.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p]
    dev = torch.device("cuda")
    res = timer_resolution(lib, dev)
    coarse = res["min_step_ns"] is None or res["min_step_ns"] > 500
    print(f"globaltimer: smallest step {res['min_step_ns']} ns, median step {res['median_step_ns']} ns "
          f"({res['ticks']} ticks in {res['reads']} back-to-back reads)")
    if coarse:
        print("globaltimer too coarse to resolve us-scale gaps: rely on the event-timed A/B")

    n, ring = args.n, 8
    g = torch.Generator(device=dev).manual_seed(0)
    xs = [torch.randn(n, 6, device=dev, generator=g) * 0.5 for _ in range(ring)]
    Xs = [torch.empty(n, 7, device=dev) for _ in range(ring)]
    ys = [torch.empty(n, 6, device=dev) for _ in range(ring)]
    key = {}
    for j in range(ring):
        key[xs[j].data_ptr()] = 2 * j
        key[Xs[j].data_ptr()] = 2 * j + 1
    side = torch.cuda.Stream()

    def seq(sp):
        for j in range(ring):
            assert lib.trace_se3_exp_fwd_f32(xs[j].data_ptr(), Xs[j].data_ptr(), n, sp) == 0
            assert lib.trace_SE3_log_fwd_f32(Xs[j].data_ptr(), ys[j].data_ptr(), n, sp) == 0

    with torch.cuda.stream(side):
        seq(ctypes.c_void_p(side.cuda_stream))
        side.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):
            seq(ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    for _ in range(5):
        graph.replay()
    torch.cuda.synchronize()
    # event-timed step with the hooks on (context for the stamps, not the headline)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(50):
        graph.replay()
    e1.record()
    torch.cuda.synchronize()
    step_us = e0.elapsed_time(e1) * 1e3 / (50 * ring)

    replays = 2
    assert lib.trace_reset() == 0
    for _ in range(replays):
        graph.replay()
    torch.cuda.synchronize()
    cap = lib.trace_capacity()
    host = np.zeros((cap, 8), dtype=np.uint64)
    cnt = lib.trace_read(host.ctypes.data_as(ctypes.POINTER(ctypes.c_ulonglong)))
    assert 0 < cnt <= cap, (cnt, cap)
    rec = host[:cnt].astype(np.int64)

    # launch index: ring position from the input pointer, replay from the order of a block's stamps
    launches = {}
    for r in rec:
        k = key[int(r[0])]
        launches.setdefault(k, []).append(r)
    rows = []
    for k in sorted(launches):
        a = np.array(launches[k])
        blk = a[:, 1] >> 32
        order = np.lexsort((a[:, 2], blk))
        a = a[order]
        rep = np.zeros(len(a), dtype=int)
        rep[1:] = (blk[order][1:] == blk[order][:-1]).astype(int)
        for i in range(1, len(a)):
            if rep[i]:
                rep[i] = rep[i - 1] + 1
        for rr in range(replays):
            rows.append((rr * 2 * ring + k, a[rep == rr]))
    rows.sort(key=lambda t: t[0])
    t_ref = min(int(a[:, 2].min()) for _, a in rows)

    out = []
    prev = None
    for idx, a in rows:
        sm = a[:, 1] & 0xFFFFFFFF
        ent, rel, land, last, ex = (a[:, 2 + i] for i in range(5))
        busy = a[:, 7] > 0
        d = {"launch": idx, "op": "Exp" if idx % 2 == 0 else "Log", "ctas": int(len(a)),
             "start_us": (int(ent.min()) - t_ref) / 1e3, "span_us": (int(ex.max()) - int(ent.min())) / 1e3}
        if prev is not None:
            pex = prev["ex"]
            d["gap_us"] = (int(land[busy].min()) - int(pex.max())) / 1e3
            d["rel_us"] = (int(rel.min()) - int(pex.max())) / 1e3
            ov = []
            for s in np.unique(sm):
                m0, m1 = prev["sm"] == s, sm == s
                if m0.any() and m1.any():
                    lo = max(int(prev["ent"][m0].min()), int(ent[m1].min()))
                    hi = min(int(pex[m0].max()), int(ex[m1].max()))
                    ov.append(max(0, hi - lo))
            d["ovl_us"] = float(np.mean(ov)) / 1e3 if ov else 0.0
            d["graph_boundary"] = idx % (2 * ring) == 0
        out.append(d)
        prev = {"ex": ex, "ent": ent, "sm": sm}

    print(f"N = {n}, ring {ring}, {replays} back-to-back replays of a {2 * ring}-launch graph; "
          f"event-timed step with hooks {step_us:.2f} us")
    print(f"{'launch':>6} {'op':>3} {'ctas':>5} {'start':>8} {'span':>7} {'gap':>7} {'rel':>7} {'ovl':>7}")
    for d in out:
        print(f"{d['launch']:>6} {d['op']:>3} {d['ctas']:>5} {d['start_us']:>8.2f} {d['span_us']:>7.2f} "
              + (f"{d['gap_us']:>7.2f} {d['rel_us']:>7.2f} {d['ovl_us']:>7.2f}" if 'gap_us' in d else "")
              + (" (graph boundary)" if d.get("graph_boundary") else ""))
    inner = [d for d in out if "gap_us" in d and not d["graph_boundary"]]
    summ = {"timer": res, "timer_too_coarse": coarse, "n": n, "step_us_hooks_on": round(step_us, 3),
            "period_us": round((out[-1]["start_us"] - out[0]["start_us"]) / (len(out) - 1), 3),
            "mean_span_us": round(float(np.mean([d["span_us"] for d in out])), 3),
            "mean_gap_us": round(float(np.mean([d["gap_us"] for d in inner])), 3),
            "mean_rel_us": round(float(np.mean([d["rel_us"] for d in inner])), 3),
            "mean_ovl_us": round(float(np.mean([d["ovl_us"] for d in inner])), 3),
            "gpu": torch.cuda.get_device_name()}
    for op in ("Exp", "Log"):
        sel = [d for d in inner if d["op"] == op]
        summ[f"mean_gap_before_{op}_us"] = round(float(np.mean([d["gap_us"] for d in sel])), 3)
    print(json.dumps(summ))
    if args.out:
        with open(args.out, "w") as f:
            json.dump({"summary": summ, "launches": out}, f, indent=1)


if __name__ == "__main__":
    sys.exit(main())

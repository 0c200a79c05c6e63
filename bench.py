#!/usr/bin/env python
"""bench.py — headline benchmark of the hot path (contract: see DESIGN.md §Measurement).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

metric  : SE3 Exp+Log Mops/s (1 op = one se3->SE3 Exp plus one SE3->se3 Log on one element)
workload: BASELINE.json configs[1] — batch 10^6, fp32, per GPU (weak scaling, no data-path collective)
step    : one Exp launch + one Log launch over one resident batch; batches rotate through a ring whose
          footprint exceeds the 126 MB L2 (Log reads the SE3 batch Exp just wrote, possibly still in L2; nothing else is).
value   : device-timed (CUDA events, max over ranks), inputs resident in HBM; W warm-up steps, then exactly K steps between
          barrier + synchronize pairs, repeated REGIONS times, median region reported.
legs    : LM step/s (PoseInv, reprojection at 1e6 / 1e7 / 2e8 residual rows, pose graph, bundle adjustment) and IMU
          Msamples/s through the public API, each with its own roofline object (bench_legs.py).
e2e     : same metric through the public API (pp.se3(...).Exp().Log()) with pinned HOST buffers,
          H2D and D2H copies inside the timed region.
outputs : --dump-outputs DIR writes rank 0's last timed step as DIR/exp_SE3.npy (n, 7) and DIR/log_se3.npy (n, 6),
          fp32, 52 MB in all; the inputs are seeded, so two builds can be compared output for output.
The reference arm (--impl reference) times the torch-CPU port of the reference's Exp/Log op
sequence (oracle/torch_port.py) on all host cores, on a bounded sample of the same workload.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

# NCCL_DEBUG=VERSION (set in the box's environment) makes NCCL print its version banner on stdout, next to the one JSON
# line this script prints.  Measured: the banner is also printed at the WARN level and ignores NCCL_DEBUG_FILE, so the
# variable is dropped (level NONE) when it only asks for the banner; any other setting of the user's is kept.
if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
    del os.environ["NCCL_DEBUG"]

import torch  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BATCH = 1_000_000
BYTES_EXP = 4 * (6 + 7)      # algorithmic bytes / element (SURVEY.md §8d): read se3 (24) + write SE3 (28)
BYTES_LOG = 4 * (7 + 6)
L2_BYTES = 126 * 2 ** 20
METRIC = "SE3 Exp+Log throughput (batch 1e6, fp32)"
UNIT = "Mops/s"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clock / throttle sampling during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); smax = float(f[1])
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax, "samples": len(sm),
                "reasons": sorted(reasons)}


def dist_setup(n_gpus):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        import datetime
        # a rank that falls out of step must fail the run in minutes, not after NCCL's default 10-minute watchdog
        dist.init_process_group("nccl", device_id=torch.device("cuda", local), timeout=datetime.timedelta(seconds=180))
    return rank, world, local


def barrier(world):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()


def max_over_ranks(ms, world, dev):
    if world > 1:
        import torch.distributed as dist
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())
    return ms


def se3_batch(n, seed, device):
    """One workload batch, the same code for both arms: tau ~ N(0,1)^3, phi = theta * axis, theta ~ U(0, pi - 0.01), axis
    uniform on the sphere (SURVEY.md §8d cfg 2)."""
    g = torch.Generator(device=device).manual_seed(seed)
    x = torch.randn(n, 6, generator=g, device=device, dtype=torch.float32)
    axis = torch.randn(n, 3, generator=g, device=device, dtype=torch.float32)
    axis = axis / axis.norm(dim=-1, keepdim=True)
    theta = torch.rand(n, 1, generator=g, device=device, dtype=torch.float32) * (3.14159265 - 0.01)
    x[:, 3:] = axis * theta
    return x.contiguous()


WORKLOAD = "SE3 Exp+Log, batch 1e6 per GPU, fp32, theta ~ U(0, pi-0.01) (BASELINE.json configs[1])"


def base_config(world):
    return {"workload": WORKLOAD, "batch_per_gpu": BATCH, "angles": "U(0, pi-0.01)",
            "parallelism": f"dp{world} (independent batches, no collective)"}


def run_ours(args):
    import pypose_b200 as pp
    from pypose_b200 import _C
    rank, world, local = dist_setup(args.gpus)
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    n = BATCH
    ring = 8                                  # 8 x 76 MB = 608 MB of distinct buffers, > 4 x L2
    xs = [se3_batch(n, 1234 + 100 * rank + j, dev) for j in range(ring)]
    Xs = [torch.empty(n, 7, device=dev) for _ in range(ring)]
    ys = [torch.empty(n, 6, device=dev) for _ in range(ring)]
    footprint = ring * n * (24 + 28 + 24)
    f_exp, f_log = _C.fn("b200_se3_exp_fwd_f32"), _C.fn("b200_SE3_log_fwd_f32")
    K, W = args.steps, max(3, args.warmup)

    def step(j, sp, which=3):
        if which & 1:
            _C.check(f_exp(ctypes.c_void_p(xs[j].data_ptr()), ctypes.c_void_p(Xs[j].data_ptr()), n, sp), "exp")
        if which & 2:
            _C.check(f_log(ctypes.c_void_p(Xs[j].data_ptr()), ctypes.c_void_p(ys[j].data_ptr()), n, sp), "log")

    side = torch.cuda.Stream(dev)

    def capture(which):
        """CUDA graphs for exactly-K replays: one graph per ring slot holding ONE step (Exp launch + Log launch) and one
        graph holding a whole trip round the ring (8 steps back to back, no host launch between them)."""
        graphs = []
        with torch.cuda.stream(side):
            for j in list(range(ring)) + [None]:
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=side):
                    spc = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
                    for jj in (range(ring) if j is None else (j,)):
                        step(jj, spc, which)
                graphs.append(g)
        torch.cuda.synchronize()
        return graphs

    with torch.cuda.stream(side):
        sp = ctypes.c_void_p(side.cuda_stream)
        for i in range(ring):
            step(i, sp)
        side.synchronize()
    graphs = capture(3)

    def timed_region(gs, k):
        """exactly k steps: k // ring trips of the 8-step graph, then k % ring single-step graphs"""
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(k // ring):
            gs[ring].replay()
        for i in range(k % ring):
            gs[i].replay()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b)

    timed_region(graphs, W)                # W untimed warm-up steps
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    regions = []
    for _ in range(REGIONS):               # each region: barrier + sync, EXACTLY K steps, sync; the median region is reported
        barrier(world)
        ms = timed_region(graphs, K)
        barrier(world)
        regions.append(max_over_ranks(ms, world, dev))
    outputs = None
    if args.dump_outputs and rank == 0:
        last = (K - 1) % ring                  # timed_region replays the ring slots in order
        outputs = {"exp_SE3": Xs[last].cpu().numpy(), "log_se3": ys[last].cpu().numpy()}
    # keep the GPU busy long enough for nvidia-smi to see clocks under load (a 0.4 ms region is shorter than one sample)
    t_end = time.perf_counter() + 0.35
    while time.perf_counter() < t_end:
        timed_region(graphs, ring * 8)
    clocks = sampler.stop() if rank == 0 else None
    regions.sort()
    ms_per_step = regions[len(regions) // 2] / K
    value = world * n / (ms_per_step * 1e-3) / 1e6

    # per-kernel durations (each kernel alone, same ring, CUDA events on the launching stream) for the roofline
    kk = (max(K, 64) + ring - 1) // ring * ring
    g_exp, g_log = capture(1), capture(2)
    for gs in (g_exp, g_log):
        timed_region(gs, ring)
    t_exp = sorted(timed_region(g_exp, kk) for _ in range(3))[1] / kk
    t_log = sorted(timed_region(g_log, kk) for _ in range(3))[1] / kk
    peak, peak_src = peaks()
    dom, t_dom, b_dom = ("se3_exp_fwd_f32", t_exp, BYTES_EXP) if t_exp >= t_log else ("SE3_log_fwd_f32", t_log, BYTES_LOG)
    ach = n * b_dom / (t_dom * 1e-3) / 1e9
    step_gbs = n * (BYTES_EXP + BYTES_LOG) / (ms_per_step * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": f"stream_kernel_tma<{dom}>", "achieved": round(ach, 1), "peak": peak,
                "unit": "GB/s", "frac": round(ach / peak, 4), "traffic": TRAFFIC.get(dom), "peak_source": peak_src,
                "bytes_per_launch": n * b_dom, "us_per_launch": round(t_dom * 1e3, 2), "exp_us": round(t_exp * 1e3, 2),
                "log_us": round(t_log * 1e3, 2), "step_gbs": round(step_gbs, 1), "step_frac": round(step_gbs / peak, 4)}

    # ---- e2e through the public API with pinned host buffers
    e2e_steps = max(32, min(256, K))
    hx = [xs[j % ring].cpu().pin_memory() for j in range(2)]
    hy = [torch.empty(n, 6).pin_memory() for _ in range(2)]
    dx = [torch.empty(n, 6, device=dev) for _ in range(2)]

    # three streams (H2D / compute / D2H) with events: PCIe is full duplex, so step i's upload, step i-1's
    # kernels and step i-2's download overlap; every byte still crosses the bus inside the timed region.
    s_in, s_out, s_c = torch.cuda.Stream(dev), torch.cuda.Stream(dev), torch.cuda.current_stream(dev)
    ev_in = [torch.cuda.Event() for _ in range(2)]
    ev_c = [torch.cuda.Event() for _ in range(2)]
    ev_out = [torch.cuda.Event() for _ in range(2)]
    dy = [None, None]

    def e2e_step(i):
        k = i % 2
        with torch.cuda.stream(s_in):
            s_in.wait_event(ev_c[k])            # dx[k] free again (its previous compute finished)
            dx[k].copy_(hx[k], non_blocking=True)
            ev_in[k].record(s_in)
        s_c.wait_event(ev_in[k])
        s_c.wait_event(ev_out[k])               # previous result in slot k has been downloaded
        dy[k] = pp.se3(dx[k]).Exp().Log().tensor()
        ev_c[k].record(s_c)
        with torch.cuda.stream(s_out):
            s_out.wait_event(ev_c[k])
            hy[k].copy_(dy[k], non_blocking=True)
            ev_out[k].record(s_out)

    for i in range(4):
        e2e_step(i)
    e2e_regions = []
    for _ in range(3):
        barrier(world)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(e2e_steps):
            e2e_step(i)
        for ev in ev_out:                      # the timed region ends when the last results have reached the host
            s_c.wait_event(ev)
        b.record()
        torch.cuda.synchronize()
        e2e_regions.append(max_over_ranks(a.elapsed_time(b), world, dev) / e2e_steps)
    e2e_ms = sorted(e2e_regions)[1]
    e2e = {"value": round(world * n / (e2e_ms * 1e-3) / 1e6, 1), "unit": UNIT, "h2d_bytes_per_step": n * 24,
           "d2h_bytes_per_step": n * 24, "ms_per_step": round(e2e_ms, 4), "steps": e2e_steps, "regions": 3,
           "api": "pp.se3(x).Exp().Log() with pinned host in/out"}

    cpu = cpu_baseline(sample_batches=10) if (rank == 0 and world == 1 and not args.no_cpu) else None
    import bench_legs
    legs = bench_legs.run(args, rank, world, dev, peak)
    if outputs is not None:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in outputs.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    if rank == 0:
        cfg = base_config(world)
        cfg.update({"launch": "CUDA graphs: K // 8 trips of an 8-step graph + K % 8 single-step graphs", "timed_regions": REGIONS,
                    "l2": f"inputs larger than L2: ring of {ring} batches, footprint {footprint >> 20} MiB > 126 MiB L2"})
        line = {"metric": METRIC, "value": round(value, 1), "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": round(ms_per_step, 6), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "gpu_launches": 2 * K}
        line.update(legs)                      # LM step/s and IMU legs, each with its own roofline (before the long keys)
        line.update({"roofline": roofline, "e2e": e2e, "cpu_baseline": cpu, "clocks": clocks, "config": cfg})
        print(json.dumps(line), flush=True)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


REGIONS = 5

# dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu --set full capture
# (profiles/); None until measured.
TRAFFIC = {}
try:
    TRAFFIC = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
except (OSError, ValueError):
    pass


def usable_cores():
    """Host threads this process may really use: affinity mask, clipped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(per) + 0.5)))
    except (OSError, ValueError):
        pass
    return n


def best_threads(fn, cores):
    """Pick the torch thread count that runs `fn` fastest (the reference's eager CPU path scales badly past
    a few dozen threads: 128 threads on the bench host were 100x slower than 16)."""
    cands = sorted({c for c in (4, 8, 16, 32, 64, cores) if c <= cores} | {cores})
    best, best_t = cands[0], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        fn()
        t = time.perf_counter(); fn(); dt = time.perf_counter() - t
        if dt < best_t:
            best, best_t = c, dt
        if dt > 4 * best_t:
            break
    torch.set_num_threads(best)
    return best


def _cpu_explog(sample_batches, warmup):
    from oracle import torch_port
    x = se3_batch(BATCH, 1234, torch.device("cpu"))
    cores = best_threads(lambda: torch_port.SE3_log(torch_port.se3_exp(x)), usable_cores())
    for _ in range(warmup):
        torch_port.SE3_log(torch_port.se3_exp(x))
    t_all = time.perf_counter()
    best = float("inf")
    for _ in range(sample_batches):
        t = time.perf_counter()
        torch_port.SE3_log(torch_port.se3_exp(x))
        best = min(best, time.perf_counter() - t)
    mean = (time.perf_counter() - t_all) / sample_batches
    return mean, best, cores


def cpu_baseline(sample_batches):
    """Reference's torch-CPU op sequence (oracle/torch_port.py) on the host cores (best thread count), plus the
    reference-side LM step and IMU integrate at the sizes the host can run (bench_legs.run_reference)."""
    import bench_legs
    mean, best, cores = _cpu_explog(sample_batches, 1)
    out = {"value": round(BATCH / mean / 1e6, 3), "unit": UNIT, "cores": cores, "kind": "port",
           "best_value": round(BATCH / best / 1e6, 3),
           "sample": f"{sample_batches} x (Exp+Log over one 1e6-element fp32 batch), torch {torch.__version__} CPU, "
                     f"{cores} threads (fastest of 4..{usable_cores()}); mean over the sample"}
    out.update(bench_legs.run_reference())
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import bench_legs
    steps = max(1, min(args.steps, 60))
    warm = max(1, min(args.warmup, 3))
    mean, best, cores = _cpu_explog(steps, warm)
    ms = mean * 1e3
    v = round(BATCH / mean / 1e6, 3)
    cfg = base_config(args.gpus)
    cfg["note"] = "each step = one full 1e6-element batch on the host; step count bounded to 60"
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "warmup": warm, "ms_per_step": round(ms, 3), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic"}
    line.update(bench_legs.run_reference())
    line.update({"cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                                  "sample": f"{steps} x Exp+Log over a 1e6 fp32 batch (oracle/torch_port.py, torch CPU)"},
                 "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "config": cfg})
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-large", dest="no_large", action="store_true", help="skip the 2e8-residual LM leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed Exp+Log step (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()

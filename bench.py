#!/usr/bin/env python
"""bench.py — headline benchmark of the learning3d_b200 hot path (contract: see DESIGN.md §5).

    python bench.py --gpus N --steps K --warmup W          # our arm (CUDA, one rank per GPU)
    python bench.py --impl reference --gpus N ...          # reference CPU path on the host cores
    python bench.py ... --dump-outputs DIR                 # also save the last timed step's kNN indices

--steps is the number of timed steps in either arm.  The inputs are seeded, so two builds run with the same
arguments can be compared output for output through --dump-outputs.

A "step" is one pass of the fused pairwise-distance + kNN kernel over one batch of BASELINE
config C2 (B=32 clouds of N=1024 points, k=20 — the DGCNN graph).  Weak scaling: every rank owns
its own B=32 batch, no data-path collective (SURVEY.md §8e).  Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

B_PER_GPU, N_PTS, K_NN = 32, 1024, 20
METRIC, UNIT = "point_pairs_per_sec", "pairs/s"
WORKLOAD = ("C2 DGCNN graph: fused pairwise-distance + top-k, B=%d clouds/GPU x N=%d pts, k=%d, fp32, "
            "int64 indices" % (B_PER_GPU, N_PTS, K_NN))
# SURVEY.md §8(d): compulsory bytes per query row = 12 B read + 8*k B int64 index write
ALG_BYTES_PER_ROW = 12 + 8 * K_NN
FLOP_PER_PAIR = 8


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000,
                    help="timed steps (the reference arm runs on the host at ~0.1-0.2 s per step: pass a few dozen)")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the ~10 s oracle timing")
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--no-graph", action="store_true", help="launch every step directly (no CUDA graph)")
    ap.add_argument("--profile", action="store_true",
                    help="for runs under ncu: no clock ramp, no CPU baseline, few secondary iterations")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the kNN indices of the last timed step to DIR/knn_idx.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    return args


def dump_outputs(directory, **arrays):
    """Save each array as DIR/<name>.npy in float64, so that two builds run with the same arguments (hence the
    same seeded inputs) can be compared output for output."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), np.asarray(a, dtype=np.float64))


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag = index, [], set(), False
        self.max_mhz = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
            nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
        }
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.002)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


def cpu_baseline_port(seconds):
    """The C oracle (OpenMP over rows) on the host cores: a bounded sample of the same workload."""
    import numpy as np
    import oracle
    rng = np.random.default_rng(1234)
    x = rng.random((B_PER_GPU, 3, N_PTS), dtype=np.float32)
    oracle.knn_expansion(x, K_NN, mt=True)          # warm-up
    reps, t0 = 0, time.perf_counter()
    while True:
        oracle.knn_expansion(x, K_NN, mt=True)
        reps += 1
        el = time.perf_counter() - t0
        if el >= seconds:
            break
    return {"value": reps * B_PER_GPU * N_PTS * N_PTS / el, "unit": UNIT,
            "cores": oracle.num_threads(), "kind": "port",
            "sample": "oracle/l3d_oracle.c knn_expansion (OpenMP), B=%d N=%d k=%d batch repeated %d x (%.1f s)"
                      % (B_PER_GPU, N_PTS, K_NN, reps, el)}


def run_reference(args, rank):
    """Reference arm: the reference's own CPU implementation of knn() (torch matmul + topk,
    utils/model_common_utils.py:3-9, restated call-for-call in oracle/ref_torch.py) on all host
    threads.  Each step is one full B=32 batch (~0.1-0.2 s)."""
    if rank != 0:
        return
    import torch
    from oracle import ref_torch
    # "all the host threads it can use": torch's intra-op pool is sized to the thread count that runs
    # this workload fastest among {all logical CPUs, half, torch's default} (oversubscribing SMT
    # siblings slows matmul + topk down), decided by one untimed call each.
    torch.manual_seed(1234)
    x = torch.rand(B_PER_GPU, 3, N_PTS)
    ncpu = os.cpu_count() or 1
    cands = sorted({ncpu, max(1, ncpu // 2), torch.get_num_threads()}, reverse=True)
    best_t, cores = None, ncpu
    for c in cands:
        torch.set_num_threads(c)
        ref_torch.knn(x, K_NN)
        t0 = time.perf_counter()
        ref_torch.knn(x, K_NN)
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best_t, cores = dt, c
    torch.set_num_threads(cores)
    steps = args.steps
    for _ in range(args.warmup):
        ref_torch.knn(x, K_NN)
    t0 = time.perf_counter()
    for _ in range(steps):
        idx = ref_torch.knn(x, K_NN)
    el = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, knn_idx=idx.numpy())
    value = steps * B_PER_GPU * N_PTS * N_PTS / el
    sample = "torch-CPU knn() restatement, %d steps of one B=%d N=%d k=%d batch, %d threads" % (
        steps, B_PER_GPU, N_PTS, K_NN, cores)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": args.warmup, "ms_per_step": 1e3 * el / steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": {"workload": WORKLOAD, "device": "host CPU, %d threads" % cores},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def run_ours(args, rank, local_rank, world):
    import torch
    from learning3d_b200 import _C

    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback)"
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    dist_on = world > 1
    if dist_on:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    lib = _C.lib()
    B, N, k = B_PER_GPU, N_PTS, K_NN

    # inputs+outputs cycled over a pool larger than L2 so no step finds its data in cache
    in_bytes, out_bytes = B * 3 * N * 4, B * N * k * 8
    pool = max(4, int(1.5 * 126e6 / (in_bytes + out_bytes)) + 1)
    torch.manual_seed(1234 + rank)
    xs = [torch.rand(B, 3, N, device=dev) for _ in range(pool)]
    outs = [torch.empty(B, N, k, dtype=torch.int64, device=dev) for _ in range(pool)]
    stream = torch.cuda.current_stream()
    sp = _C._P(stream.cuda_stream)
    null = _C._P(None)

    def step(i, sptr=None):
        j = i % pool
        rc = lib.l3d_knn_expansion(_C._P(xs[j].data_ptr()), B, N, k, _C._P(outs[j].data_ptr()), null,
                                   sptr if sptr is not None else sp)
        if rc:
            _C.check(rc, "knn")

    # clock ramp (untimed) + the W warm-up steps
    t0 = time.perf_counter()
    i = 0
    while not args.profile and time.perf_counter() - t0 < 0.3:
        for _ in range(50):
            step(i); i += 1
        torch.cuda.synchronize()
    for w in range(max(args.warmup, 3)):
        step(w)
    torch.cuda.synchronize()

    # The step is a ~30 us launch: capture one pass over the buffer pool (min(pool, steps) launches of
    # our kernel, nothing else) in a CUDA graph and replay it, so the timed region measures the kernel and
    # not the per-launch driver gap.  Steps that do not fill a whole replay are launched directly.
    graph, per_replay = None, min(pool, max(1, args.steps))
    if not args.no_graph and not args.profile and args.steps >= 4:
        side = torch.cuda.Stream()
        side.wait_stream(stream)
        with torch.cuda.stream(side):
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=side):
                cap = _C._P(torch.cuda.current_stream().cuda_stream)
                for s in range(per_replay):
                    step(s, cap)
        stream.wait_stream(side)
        for _ in range(3):
            graph.replay()
        torch.cuda.synchronize()
    replays = (args.steps // per_replay) if graph is not None else 0
    direct = args.steps - replays * per_replay

    sampler = ClockSampler(local_rank)
    sampler.start()
    if dist_on:
        dist.barrier()
    torch.cuda.synchronize()
    l0 = _C.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(replays):
        graph.replay()
    for s in range(direct):
        step(s)
    e1.record(stream)
    torch.cuda.synchronize()
    # kernels of ours executed in the timed region: graph nodes replayed + direct launches
    launches = replays * per_replay + (_C.launch_count() - l0)
    ms = e0.elapsed_time(e1)
    # the buffer the last timed step wrote: the last direct launch, else the last node of the graph
    last_idx = outs[(direct - 1) % pool if direct else per_replay - 1].cpu() if args.dump_outputs else None
    if dist_on:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.barrier()
        ms = float(t.item())
    sampler.stop_flag = True
    sampler.join(timeout=1.0)

    # ---- end-to-end through the host-buffer C ABI (pinned host memory, copies inside) -----
    e2e_steps = 3 if args.profile else max(10, min(args.steps, 200))
    hx = torch.rand(B, 3, N).pin_memory()
    hidx = torch.empty(B, N, k, dtype=torch.int64).pin_memory()
    for _ in range(3):
        _C.check(lib.l3d_knn_expansion_host(_C._P(hx.data_ptr()), B, N, k, _C._P(hidx.data_ptr())), "e2e")
    if dist_on:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        rc = lib.l3d_knn_expansion_host(_C._P(hx.data_ptr()), B, N, k, _C._P(hidx.data_ptr()))
        if rc:
            _C.check(rc, "e2e")
    e2e_s = time.perf_counter() - t0
    if dist_on:
        t = torch.tensor([e2e_s], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())

    extra = {}
    # the timed region above is K launches (~0.7 ms at K = 20): also report the same step over a >= 0.5 s window
    if graph is not None and not args.profile:
        n_rep = max(1, int(0.5 / max(1e-6, per_replay * ms * 1e-3 / max(1, args.steps))))
        w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0.record(stream)
        for _ in range(n_rep):
            graph.replay()
        w1.record(stream)
        torch.cuda.synchronize()
        wms = w0.elapsed_time(w1)
        extra["knn_window"] = {"steps": n_rep * per_replay, "seconds": wms * 1e-3,
                               "us_per_step": wms * 1e3 / (n_rep * per_replay),
                               "pairs_per_sec_per_gpu": B * N * N * n_rep * per_replay / (wms * 1e-3)}
    try:
        extra.update(chamfer_bench(torch, dev, dist_on, world, 5 if args.profile else 200))
    except ImportError:
        pass
    if world == 1:
        extra.update(tensor_core_bench(torch, dev, 2 if args.profile else 30))
    if not args.profile:
        extra["configs"] = config_rows(torch, dev, lib, world, rank, dist_on)

    if rank == 0:
        pairs_per_step = world * B * N * N
        value = pairs_per_step * args.steps / (ms * 1e-3)
        kernel_s = ms * 1e-3 / args.steps
        peak, peak_src = peaks()
        alg_bytes = B * N * ALG_BYTES_PER_ROW
        achieved = alg_bytes / kernel_s / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "parallelism": "batch-shard dp%d (no data-path collective)" % world,
                       "global_batch": world * B,
                       "launch": ("cuda-graph replay (%d launches per graph) + %d direct" % (per_replay, direct)
                                  if graph is not None else "direct launches"),
                       "l2": "inputs+outputs cycled over a %d-buffer pool = %.0f MB > 126 MB L2"
                             % (pool, pool * (in_bytes + out_bytes) / 1e6)},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": ncu_traffic(),
                         "peak_source": peak_src, "kernel": "l3d::knn_duo_kernel<PPG=8,k=20> (knn_tpr.cu: thread-per-row selection, two warps per 64 rows)",
                         "algorithmic_bytes_per_launch": alg_bytes,
                         "fp32_gflops_achieved": B * N * N * FLOP_PER_PAIR / kernel_s / 1e9,
                         "note": "fp32-issue/selection bound once the NxN matrix is not materialised "
                                 "(SURVEY.md §8d): a perfect kernel reaches ~20% of HBM peak at this shape; the fma "
                                 "floor of the two candidate passes is 8.3 us (DESIGN.md §3.1)"},
            "e2e": {"value": world * B * N * N * e2e_steps / e2e_s, "unit": UNIT,
                    "h2d_bytes_per_step": in_bytes, "d2h_bytes_per_step": B * N * k * 2,
                    "ms_per_step": 1e3 * e2e_s / e2e_steps,
                    "path": "l3d_knn_expansion_host: host fp32 cloud in, host int64 indices out; H2D, kernel and D2H "
                            "inside (indices cross PCIe as uint16 and are widened to the caller's int64 array by "
                            "host threads while later slices are in flight), one sync"},
            "gpu_launches": launches,
            "clocks": sampler.summary(),
        }
        if extra:
            line["extra"] = extra
        if world == 1 and not args.no_cpu_baseline and not args.profile:
            line["cpu_baseline"] = cpu_baseline_port(args.cpu_seconds)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, knn_idx=last_idx.numpy())
        print(json.dumps(line), flush=True)
    if dist_on:
        dist.destroy_process_group()


def ncu_traffic():
    """dram bytes per launch of the kNN kernel from the committed ncu capture (profiles/), or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "knn_traffic.json")) as f:
            return json.load(f)["dram_bytes_per_launch"]
    except Exception:
        return None


def chamfer_bench(torch, dev, dist_on, world, iters=200):
    """Secondary metric of BASELINE.json: Chamfer fwd+bwd clouds/s (config C1 shape per GPU and a
    B=32 batch), through the public ChamferDistanceLoss API."""
    from learning3d_b200.losses import ChamferDistanceLoss
    crit = ChamferDistanceLoss()
    out = {}
    for B in (4, 32):
        a = torch.rand(B, 1024, 3, device=dev, requires_grad=True)
        b = torch.rand(B, 1024, 3, device=dev, requires_grad=True)
        for _ in range(min(10, iters)):
            a.grad = b.grad = None
            crit(a, b).backward()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            a.grad = b.grad = None
            crit(a, b).backward()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / iters
        if dist_on:
            import torch.distributed as dist
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        out["chamfer_fwd_bwd_clouds_per_sec_B%d" % B] = world * B / (ms * 1e-3)
        out["chamfer_fwd_bwd_ms_B%d" % B] = ms
    return out


def _events_ms(torch, fn, iters, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def _tf32_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["bf16_tflops"]) / 2.0, "half of the measured dense bf16 cuBLAS rate (MEASURED_PEAKS.json)"
    except Exception:
        return 1125.0, "nominal dense TF32 (B200_PROFILING.md)"


def config_rows(torch, dev, lib, world, rank, dist_on):
    """BASELINE.json's other configurations as secondary rows (per rank; rank 0 reports its own numbers):
    C1 Chamfer fwd+bwd, C2 whole DGCNN forward, C3 DCP forward, C4 FlowNet3D forward, C5 EMD fwd+bwd — each
    with the algorithmic work SURVEY.md §8(d) fixes and, where it is cheap, the reference beside it."""
    from learning3d_b200 import _C
    rows = {}
    hbm, _ = peaks()
    tf32_peak, tf32_src = _tf32_peak()
    P = lambda t: _C._P(t.data_ptr())

    # ---- C1: Chamfer fwd+bwd on two [4,1024,3] clouds ------------------------------------------------------
    Bc, n = 4, 1024
    a = torch.rand(Bc, n, 3, device=dev); b = torch.rand(Bc, n, 3, device=dev)
    d1 = torch.empty(Bc, n, device=dev); d2 = torch.empty(Bc, n, device=dev)
    i1 = torch.empty(Bc, n, dtype=torch.int32, device=dev); i2 = torch.empty(Bc, n, dtype=torch.int32, device=dev)
    loss = torch.empty(1, device=dev); one = torch.ones(1, device=dev)
    ws = torch.empty(int(lib.l3d_chamfer_ws_bytes(Bc, n, n)), dtype=torch.uint8, device=dev)
    g1 = torch.empty_like(a); g2 = torch.empty_like(b)

    def chamfer_step(sp):
        _C.check(lib.l3d_chamfer_loss_forward(P(a), P(b), Bc, n, n, P(d1), P(d2), P(i1), P(i2), P(loss), P(ws), sp))
        _C.check(lib.l3d_chamfer_loss_backward(P(a), P(b), Bc, n, n, P(d1), P(d2), P(i1), P(i2), P(one), P(g1), P(g2), sp))
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            chamfer_step(_C._P(side.cuda_stream))
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr, stream=side):
            cap = _C._P(torch.cuda.current_stream().cuda_stream)
            for _ in range(20):
                chamfer_step(cap)
    torch.cuda.current_stream().wait_stream(side)
    ms = _events_ms(torch, gr.replay, 20) / 20
    ha, hb = torch.rand(Bc, n, 3).pin_memory(), torch.rand(Bc, n, 3).pin_memory()
    hl = torch.empty(1).pin_memory(); hg1 = torch.empty(Bc, n, 3).pin_memory(); hg2 = torch.empty(Bc, n, 3).pin_memory()
    host = lambda: _C.check(lib.l3d_chamfer_loss_fwd_bwd_host(P(ha), P(hb), Bc, n, n, P(hl), P(hg1), P(hg2)))
    for _ in range(3):
        host()
    t0 = time.perf_counter()
    for _ in range(200):
        host()
    host_s = (time.perf_counter() - t0) / 200
    alg = 425984                                       # SURVEY.md §8(d): bytes per C1 fwd+bwd
    rows["C1_chamfer_fwd_bwd"] = {
        "workload": "Chamfer loss fwd+bwd, two [4,1024,3] clouds, fp32 (2 launches)",
        "value": Bc / (ms * 1e-3), "unit": "clouds/s", "us_per_step": ms * 1e3, "timing": "CUDA-graph replay of 20 fwd+bwd pairs",
        "e2e": {"value": Bc / host_s, "unit": "clouds/s", "us_per_step": host_s * 1e6,
                "h2d_bytes_per_step": 2 * Bc * n * 12, "d2h_bytes_per_step": 2 * Bc * n * 12 + 4,
                "path": "l3d_chamfer_loss_fwd_bwd_host (pinned host buffers)"},
        "roofline": {"bound": "hbm", "achieved": alg / (ms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                     "frac": alg / (ms * 1e-3) / 1e9 / hbm, "algorithmic_bytes_per_step": alg,
                     "note": "8.4 M pair evaluations on 425 KB: latency / issue bound, not HBM bound"},
    }
    if world == 1:
        import numpy as np
        import oracle
        an, bn = a.cpu().numpy(), b.cpu().numpy()
        oracle.chamfer_loss(an, bn)
        t0, reps = time.perf_counter(), 0
        while time.perf_counter() - t0 < 2.0:
            oracle.chamfer_loss(an, bn); reps += 1
        el = time.perf_counter() - t0
        rows["C1_chamfer_fwd_bwd"]["cpu_baseline"] = {
            "value": Bc * reps / el, "unit": "clouds/s (forward only)", "cores": 1, "kind": "port",
            "sample": "oracle/l3d_oracle.c chamfer (nnsearch restatement, single thread like the reference's C++), %d x" % reps}

    # ---- C2: whole DGCNN forward (kNN graph + EdgeConv stack + conv5), eval ---------------------------------------
    from learning3d_b200.models import DCP, DGCNN
    Bd, N, k, emb = B_PER_GPU, N_PTS, K_NN, 512
    net = DGCNN(emb_dims=emb).to(dev).eval()
    x = torch.rand(Bd, N, 3, device=dev)
    with torch.no_grad():
        ms = _events_ms(torch, lambda: net(x), 20)
        flop = 2.0 * Bd * N * k * (6 * 64 + 64 * 64 + 64 * 128 + 128 * 256) + 2.0 * Bd * N * 512 * emb
        issued = 3.0 * (flop - 2.0 * Bd * N * k * 6 * 64) / (ms * 1e-3) / 1e12
        row = {"workload": "DGCNN(emb 512).forward eval: kNN graph + EdgeConv x4 + conv5, B=32 N=1024 k=20, fp32 (3xTF32 on tcgen05)",
               "value": Bd / (ms * 1e-3), "unit": "clouds/s", "us_per_step": ms * 1e3, "launches_per_step": 6,
               "roofline": {"bound": "tensor", "achieved": issued, "peak": tf32_peak, "unit": "TFLOP/s",
                            "frac": issued / tf32_peak, "peak_source": tf32_src,
                            "note": "issued TF32 MMA rate (3 MMAs per fp32-equivalent product); fp32-equivalent = achieved / 3"}}
        if world == 1:
            from oracle import ref_torch
            xt = x.permute(0, 2, 1).contiguous()

            def torch_gpu():
                h, pooled = ref_torch.get_graph_feature(xt, k=k), []
                for i in range(1, 5):
                    h = torch.relu(getattr(net, "bn%d" % i)(getattr(net, "conv%d" % i)(h)))
                    pooled.append(h.max(dim=-1, keepdim=True)[0])
                return torch.relu(net.bn5(net.conv5(torch.cat(pooled, 1))))
            torch.backends.cudnn.allow_tf32 = False
            row["reference_torch_ops_same_gpu_fp32_us"] = _events_ms(torch, torch_gpu, 5, 2) * 1e3
            torch.backends.cudnn.allow_tf32 = True
            row["reference_torch_ops_same_gpu_tf32_us"] = _events_ms(torch, torch_gpu, 5, 2) * 1e3
            torch.backends.cudnn.allow_tf32 = False
            cnet = DGCNN(emb_dims=emb).eval()
            cnet.load_state_dict(net.state_dict())
            xc = xt.cpu()

            def torch_cpu():
                h, pooled = ref_torch.get_graph_feature(xc, k=k), []
                for i in range(1, 5):
                    h = torch.relu(getattr(cnet, "bn%d" % i)(getattr(cnet, "conv%d" % i)(h)))
                    pooled.append(h.max(dim=-1, keepdim=True)[0])
                return torch.relu(cnet.bn5(cnet.conv5(torch.cat(pooled, 1))))
            torch_cpu()
            t0 = time.perf_counter()
            for _ in range(3):
                torch_cpu()
            el = (time.perf_counter() - t0) / 3
            row["cpu_baseline"] = {"value": Bd / el, "unit": "clouds/s", "cores": torch.get_num_threads(), "kind": "port",
                                   "sample": "reference layer sequence in torch on the host, 3 x one B=32 batch"}
        rows["C2_dgcnn_forward"] = row

        # ---- C3: DCP forward (DGCNN-512 + Transformer + SVDHead, cycle) -------------------------------------------
        dcp = DCP(feature_model=DGCNN(emb_dims=512), cycle=True).to(dev).eval()
        Bs = max(1, Bd // world) if dist_on else Bd          # strong scaling: global B = 32 sharded over the ranks
        tpl = torch.rand(Bs, N, 3, device=dev); src = torch.rand(Bs, N, 3, device=dev)

        def dcp_step():
            out = dcp(tpl, src)
            val = out["est_t"].square().sum()
            if dist_on:
                import torch.distributed as dist
                dist.all_reduce(val)                          # the size-weighted loss reduction of dist.py:32-44
            return val
        ms = _events_ms(torch, dcp_step, 5, 2)
        if dist_on:
            import torch.distributed as dist
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        rows["C3_dcp_forward"] = {
            "workload": "DCP(DGCNN-512 + Transformer + SVDHead, cycle).forward eval, global B=%d (B=%d per rank), N=1024, fp32"
                        % (Bs * world, Bs),
            "value": Bs * world / (ms * 1e-3), "unit": "pairs/s", "us_per_step": ms * 1e3,
            "scaling": "strong" if dist_on else "single GPU", "collective": "one all-reduce(sum) of the scalar inside the step" if dist_on else None}

    if world == 1:
        with torch.no_grad():
            # ---- C4: FlowNet3D forward ----------------------------------------------------------------------------
            from learning3d_b200.models import FlowNet3D
            fn = FlowNet3D().to(dev).eval()
            pc1 = torch.rand(16, 3, 2048, device=dev) * 4 - 2
            pc2 = pc1 + 0.05 * torch.randn_like(pc1)
            f1 = torch.rand(16, 3, 2048, device=dev); f2 = torch.rand(16, 3, 2048, device=dev)
            ms = _events_ms(torch, lambda: fn(pc1, pc2, f1, f2), 5, 2)
            rows["C4_flownet3d_forward"] = {"workload": "FlowNet3D.forward eval, B=16 N=2048, set-conv grouping on libl3d_b200.so",
                                            "value": 16 / (ms * 1e-3), "unit": "cloud pairs/s", "us_per_step": ms * 1e3}
        # ---- C5: EMD fwd (+bwd) B=8 N=1024 ----------------------------------------------------------------------
        e1 = torch.rand(8, 1024, 3, device=dev); e2 = torch.rand(8, 1024, 3, device=dev)
        cost = torch.empty(8, device=dev); match = torch.empty(8, 1024, 1024, device=dev)
        wsf = torch.empty(int(lib.l3d_emd_forward_ws_bytes(8, 1024, 1024)), dtype=torch.uint8, device=dev)
        wsb = torch.empty(int(lib.l3d_emd_backward_ws_bytes(8, 1024, 1024)), dtype=torch.uint8, device=dev)
        gg1 = torch.empty_like(e1); gg2 = torch.empty_like(e2)
        st = _C.stream()
        fwd = lambda: _C.check(lib.l3d_emd_forward(P(e1), P(e2), 8, 1024, 1024, P(cost), P(match), P(wsf), st))
        bwd = lambda: _C.check(lib.l3d_emd_backward(P(e1), P(e2), P(match), 8, 1024, 1024, P(gg1), P(gg2), P(wsb), st))
        ms_f = _events_ms(torch, fwd, 20)
        ms_b = _events_ms(torch, bwd, 20)
        exps = 251658240.0                                 # SURVEY.md §8(d): exp-weighted pair evaluations, forward
        rows["C5_emd"] = {"workload": "approximate EMD B=8 N=1024 (10 levels), forward = persistent sweep launch + match/cost launch",
                          "value": 8 / ((ms_f + ms_b) * 1e-3), "unit": "clouds/s (fwd+bwd)", "forward_us": ms_f * 1e3,
                          "backward_us": ms_b * 1e3,
                          "roofline": {"bound": "mufu", "achieved": (exps + 10 * 8 * 1024 * 1024) / (ms_f * 1e-3) / 1e12,
                                       "peak": 148 * 16 * 1.965e9 / 1e12, "unit": "T ex2/s",
                                       "note": "ex2.approx issue rate (16 / clk / SM); forward only"}}
    return rows


def tensor_core_bench(torch, dev, iters=30):
    """Tensor-core rows of the path (per GPU, not aggregated): DCP SVD-head front half at C3
    (B=32, d_k=512, N=1024; svd.py:23-28 fused) and the feature-space kNN graph (B=32, C=64, N=1024, k=20)."""
    from learning3d_b200.utils import knn
    from learning3d_b200.utils.svd import soft_correspondence
    out = {}
    es = torch.randn(32, 512, 1024, device=dev)
    et = torch.randn(32, 512, 1024, device=dev)
    tg = torch.rand(32, 3, 1024, device=dev)
    xf = torch.randn(32, 64, 1024, device=dev)
    for name, fn, flop in (("svd_head_front_C3", lambda: soft_correspondence(es, et, tg), 2.0 * 32 * 1024 * 1024 * 512),
                           ("knn_features_C64", lambda: knn(xf, 20), None)):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / iters
        out[name + "_us"] = ms * 1e3
        if flop:
            out[name + "_fp32_equiv_tflops"] = flop / (ms * 1e-3) / 1e12
            # tensor-pipe view: 3xTF32 issues three TF32 MMAs per fp32-equivalent product; the TF32 peak is
            # taken as half of the measured dense bf16 cuBLAS throughput (MEASURED_PEAKS.json)
            issued = 3.0 * flop / (ms * 1e-3) / 1e12
            out[name + "_issued_tf32_tflops"] = issued
            try:
                with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                    out[name + "_frac_of_measured_tf32_peak"] = issued / (float(json.load(f)["bf16_tflops"]) / 2.0)
            except Exception:
                pass
    return out


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()

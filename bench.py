#!/usr/bin/env python
"""bench.py — Gaussians->voxels throughput of the splat hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

A step is one forward pass of the splat op (pack + supertile lists + render; 3 kernel launches, replayed from a CUDA
graph) over one synthetic sample of BASELINE.json configs[1]: `nuscenes_gs25600_solid.py` shape — 25 600 Gaussians
(+ the "empty" Gaussian) into the 200x200x16 grid, 18 classes, batch 1 per GPU.  Prints ONE JSON line (rank 0).
Keys follow the driver contract; see DESIGN.md "Measurement".

* value        whole-job Gaussians/s with inputs resident in HBM, CUDA-event timed, max over ranks
* e2e          the same metric through the drop-in module call `local_aggregate.LocalAggregator.forward` with HOST
               (pinned) inputs: H2D of every input + forward + arg-max + D2H of the occupancy prediction inside the
               timed region; `h2d_floor_ms` is the plain pinned copy of the same bytes on the same box
* roofline     the tile render kernel timed alone (events recorded around it inside the C ABI, debug header),
               algorithmic bytes 112*G + 84*N (SURVEY.md §8d) over the measured HBM copy peak; `roofline_cfg3` is the
               same figure for BASELINE config 3 (144 000 Gaussians)
* fwd_bwd      BASELINE config 5: forward + backward at 4 samples per GPU in ONE batched launch per kernel, one scalar
               loss all-reduce per step
* prob         BASELINE config 4: probabilistic head, 6 400 Gaussians, 2 samples per GPU (bs 4 over 2 GPUs), both roofs
* cpu_baseline the oracle's C/OpenMP port of the reference algorithm on the host cores (rank 0)

`--impl reference` times that CPU port as the reference arm (the reference has no CPU implementation of the splat; its
CUDA op cannot run without a GPU build of torch extensions — when oracle/_ref was shipped, its timing on this GPU is
reported as `ref_cuda_op` in the main line).  It always runs on ONE host CPU (rank 0), whatever --gpus says.

`--dump-outputs DIR` writes what the timed path returned in its last timed step (rank 0) as DIR/logits.npy, the
[N, 18] float32 logits (46 MB).  The inputs are seeded, so two builds run with the same arguments can be compared
output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOAD = "gs25600_solid"
METRIC = "gaussians_to_voxels_per_sec"
UNIT = "Gaussians/s"
G_COUNTED = 25600                 # learned Gaussians per sample (the empty one is overhead)
N_SETS = 6                        # rotating input/output sets so the working set exceeds L2
FP32_PEAK_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12   # CUDA-core fp32 roof of a B200: 148 SMs x 128 FMA lanes x 2 x 1.965 GHz


def _algorithmic_bytes(G, N, C=18, prob=False):
    # SURVEY.md §8d: inputs read once + outputs written once.  base 112*G + 84*N, prob 112*G + 96*N (C = 18)
    return (3 + 6 + 1 + C) * 4 * G + 12 * N + 4 * (C + (3 if prob else 0)) * N


def _algorithmic_bytes_bwd(G, N, C=18, prob=False):
    # base 224*G + 84*N, prob 224*G + 172*N
    return 2 * (3 + 6 + 1 + C) * 4 * G + 12 * N + (4 * (2 * C + 4) * N if prob else 4 * C * N)


def _config(world, perturb):
    """The `config` object of the JSON line — the SAME dict for both arms (the driver compares them)."""
    return {"workload": f"{WORKLOAD}: 25600 Gaussians (+1 empty) -> 200x200x16x18 voxels, batch 1 per GPU, points = "
                        + ("perturbed voxel centres" if perturb else "voxel centres (BASELINE.md §3)"),
            "l2": f"{N_SETS} rotating input/output/workspace sets (> 126 MB L2)",
            "parallelism": f"dp{world} (one sample per GPU, scalar loss all-reduce)"}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons sampled while the timed region runs."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self._stop_evt = index, [], set(), threading.Event()
        self.max_mhz = None

    def run(self):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [p.strip() for p in out.strip().split(",")]
                self.samples.append(float(parts[0]))
                self.max_mhz = float(parts[1])
                for n, v in zip(names, parts[3:7]):
                    if v.lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                pass
            self._stop_evt.wait(0.1)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=10)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


def _bind_to_gpu_numa_node(index):
    """Pin this process to the CPUs NVML reports as local to the GPU, so that the pinned host
    buffers of the e2e leg are first-touched on the GPU's NUMA node (a remote node can cut the H2D
    rate several-fold).  Best effort: returns a short description or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = [64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1]
        if cpus:
            os.sched_setaffinity(0, cpus)
            return f"{len(cpus)} cpus local to gpu {index}"
    except Exception:
        pass
    return None


def _measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return float(json.load(open(path))["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


def _cpu_port_once(kw, inp):
    """One forward of the CPU port (oracle C code, all OpenMP threads).  Returns seconds."""
    import oracle
    a = {k: v[0].numpy() for k, v in inp.items()}
    dims = (kw["H"], kw["W"], kw["D"])
    t0 = time.perf_counter()
    pi, mi, radii = oracle.host_prep(a["pts"], a["means"], a["scales"], kw["pc_min"], kw["grid_size"],
                                     kw["scale_multiplier"])
    cov6 = oracle.cov6_from_3x3(a["cov"])
    out, pairs = oracle.splat_forward(a["pts"], pi, a["means"], mi, a["opa"], a["sem"], cov6, radii, dims, "f32")
    sec = time.perf_counter() - t0
    _LAST_PORT["logits"], _LAST_PORT["pairs"] = out, int(pairs)
    return sec


_LAST_PORT = {}   # logits / (voxel, Gaussian) pair count of the most recent CPU-port forward (checker side figures)


def _all_host_threads():
    """Give the CPU port every core this process may run on, whatever OMP_NUM_THREADS a launcher (torchrun sets 1)
    exported.  Returns the thread count in effect."""
    import oracle
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    return oracle.set_num_threads(n)


def _dump_outputs(outdir, arrays):
    """--dump-outputs: each array as <outdir>/<name>.npy, float32."""
    import numpy as np
    os.makedirs(outdir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(outdir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float32))


def run_reference_arm(args):
    """Reference arm: the reference algorithm's CPU port on this box's host cores.  ONE host CPU at any --gpus:
    under torchrun rank 0 alone runs and prints it, the other ranks exit without work."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from gaussianformer_b200.synthetic import make_splat_inputs
    cores = _all_host_threads()
    kw, inp, _ = make_splat_inputs(WORKLOAD, seed=0, perturb=args.perturb)
    for _ in range(min(max(args.warmup, 1), 3)):       # the port has no clocks or caches to warm beyond a few passes
        _cpu_port_once(kw, inp)
    steps = args.steps
    t = [_cpu_port_once(kw, inp) for _ in range(steps)]
    if args.dump_outputs:
        _dump_outputs(args.dump_outputs, {"logits": _LAST_PORT["logits"]})
    sec = sum(t) / len(t)
    value = G_COUNTED / sec
    sample = (f"{steps} full forward passes of the {WORKLOAD} sample (N=640000 points, G=25601), {sec:.3f} s each; "
              f"one host CPU ({cores} OpenMP threads) regardless of --gpus")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": steps, "warmup": max(args.warmup, 3), "ms_per_step": sec * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": _config(args.gpus, args.perturb),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-extras", action="store_true", help="skip the side measurements (bwd, DAF, ref op) and the config 3/4/5 legs")
    ap.add_argument("--no-graph", action="store_true", help="launch the three kernels of a step directly instead of replaying a CUDA graph")
    ap.add_argument("--perturb", action="store_true", help="jitter every point inside its voxel (LoadOccupancySurroundOcc(perturb=True)); "
                    "the shipped configs and BASELINE.md use exact voxel centres")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference_arm(args)

    import torch
    import torch.distributed as dist
    from gaussianformer_b200 import _lib
    from gaussianformer_b200.splat import _make_desc, _ptr, LocalAggregator
    from gaussianformer_b200.synthetic import make_splat_inputs
    import ctypes

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback of the product path)"
    torch.cuda.set_device(local_rank)
    numa = _bind_to_gpu_numa_node(local_rank)   # pinned staging buffers must live next to the GPU
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    L = _lib.lib()
    W = max(args.warmup, 3)
    K = args.steps

    # ---- resident inputs: N_SETS different samples (seeded), rotated so no step re-reads L2 -------
    PERTURB = args.perturb
    kw, inp0, _ = make_splat_inputs(WORKLOAD, seed=rank * 100, perturb=PERTURB)
    sets = []
    for i in range(N_SETS):
        _, inp, _ = (kw, inp0, None) if i == 0 else make_splat_inputs(WORKLOAD, seed=rank * 100 + i, perturb=PERTURB)
        t = {k: v[0].to(dev).contiguous() for k, v in inp.items()}
        t["cov"] = t["cov"].reshape(-1, 9).contiguous()
        sets.append(t)
    G, N, C = sets[0]["means"].shape[0], sets[0]["pts"].shape[0], 18
    desc = _make_desc(G, N, C, kw["H"], kw["W"], kw["D"], _lib.GF_SPLAT_BASE, 1, 9, kw["pc_min"], kw["grid_size"],
                      float(kw["scale_multiplier"]), 0)
    ws_bytes = L.gf_splat_forward_workspace_bytes(ctypes.byref(desc))
    outs = [torch.empty((N, C), device=dev) for _ in range(N_SETS)]
    wss = [torch.empty(ws_bytes, dtype=torch.uint8, device=dev) for _ in range(N_SETS)]
    stream = torch.cuda.current_stream(dev)
    calls = []
    for t, o, w in zip(sets, outs, wss):
        ins = _lib.SplatInputs(_ptr(t["pts"]), None, _ptr(t["means"]), None, _ptr(t["opa"]), _ptr(t["sem"]),
                               _ptr(t["cov"]), None, _ptr(t["scales"]))
        ou = _lib.SplatOutputs(_ptr(o), None, None, None, None)
        calls.append((ins, ou, w))
    loss_buf = torch.zeros(1, device=dev)
    pending = []

    def direct_call(i, s):
        ins, ou, w = calls[i % N_SETS]
        _lib.check(L.gf_splat_forward(ctypes.byref(desc), ctypes.byref(ins), ctypes.byref(ou), _ptr(w), ws_bytes,
                                      ctypes.c_void_p(s.cuda_stream)))

    # One CUDA graph per resident set: pack -> list -> render with their programmatic-dependent-launch edges, so that
    # a step costs one graph launch and `value` does not depend on how fast the host issues three launches.
    graphs = None
    if not args.no_graph:
        try:
            for i in range(N_SETS):
                direct_call(i, stream)                      # warm (module load, attribute caches) before capturing
            torch.cuda.synchronize(dev)
            graphs = []
            cap_stream = torch.cuda.Stream(dev)
            for i in range(N_SETS):
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=cap_stream):
                    direct_call(i, torch.cuda.current_stream(dev))
                graphs.append(g)
        except Exception as e:                              # fall back to direct launches, and say so
            graphs = None
            print(f"[bench] CUDA graph capture failed ({e!r}); using direct launches", file=sys.stderr)
            torch.cuda.synchronize(dev)

    def step(i):
        if graphs is not None:
            graphs[i % N_SETS].replay()
        else:
            direct_call(i, stream)
        if world > 1:
            # north star: NCCL only for the (scalar) loss all-reduce.  It is issued asynchronously on
            # NCCL's stream so that it overlaps the next sample's kernels; every handle is waited for
            # before the timed region closes.
            pending.append(dist.all_reduce(loss_buf, async_op=True))
            if len(pending) > 8:
                pending.pop(0).wait()

    def timed_region(nsteps, fn):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for i in range(nsteps):
            fn(i)
        while pending:
            pending.pop(0).wait()
        e1.record(stream)
        torch.cuda.synchronize(dev)
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            dist.barrier()
        return float(ms.item())

    for i in range(W):
        step(i)
    sampler = ClockSampler(local_rank)
    sampler.start()
    total_ms = timed_region(K, step)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        _dump_outputs(args.dump_outputs, {"logits": outs[(K - 1) % N_SETS].cpu().numpy()})
    ms_per_step = total_ms / K
    value = world * G_COUNTED / (ms_per_step * 1e-3)

    # ---- roofline: the render kernel alone, events recorded around it inside the C ABI -----------
    peak, peak_kind = _measured_peak()

    def render_alone(call, nrep):
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(nrep)]
        for i, (a, b) in enumerate(evs):
            a.record(stream); b.record(stream)          # materialise the underlying cudaEvent_t
            L.gf_debug_set_render_events(ctypes.c_void_p(a.cuda_event), ctypes.c_void_p(b.cuda_event))
            call(i)
        L.gf_debug_set_render_events(None, None)
        torch.cuda.synchronize(dev)
        ms = sorted(a.elapsed_time(b) for a, b in evs)
        return sum(ms) / len(ms)

    render_ms = render_alone(lambda i: direct_call(i, stream), min(max(K, 10), 50))
    alg = _algorithmic_bytes(G, N, C)
    achieved = alg / (render_ms * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "render_traffic.json")
    if os.path.exists(tpath):
        traffic = json.load(open(tpath)).get("dram_bytes_per_launch")
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "kernel": "render_tile_kernel<18,false>", "kernel_ms": render_ms,
                "algorithmic_bytes": alg, "peak_source": peak_kind + " (MEASURED_PEAKS.json hbm_gbs, burst copy)"}

    # ---- e2e: the drop-in module call, HOST inputs: H2D + forward + arg-max + D2H every step ----
    # Each sample's six input tensors live in ONE pinned staging buffer (what a collate function
    # would produce), so a step is one H2D copy, the module call, and one D2H copy of the occupancy
    # prediction.  The host consumes prediction i-1 while step i is in flight (two result buffers),
    # i.e. copies and kernels of consecutive steps overlap CPU work but every step's copies are
    # inside the timed region.
    module = LocalAggregator(**kw).to(dev)
    module.validate = False     # the D2H read of the prediction is the step's synchronisation point
    n_host = 3

    def stage(keys):
        layouts, host = [], []
        for i in range(n_host):
            inp = inp0 if i == 0 else make_splat_inputs(WORKLOAD, seed=rank * 100 + i, perturb=PERTURB)[1]
            offs, off = {}, 0
            for k in keys:
                v = inp[k]
                offs[k] = (off, v.numel(), tuple(v.shape))
                off += (v.numel() + 63) // 64 * 64          # 256-byte aligned slices
            buf = torch.empty(off, dtype=torch.float32).pin_memory()
            for k in keys:
                o, nel, _ = offs[k]
                buf[o:o + nel].copy_(inp[k].reshape(-1))
            layouts.append(offs)
            host.append(buf)
        return layouts, host

    pred_host = [torch.empty(N, dtype=torch.uint8).pin_memory() for _ in range(2)]
    done = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [0]
    copy_stream = torch.cuda.Stream(dev)
    h2d_done = [torch.cuda.Event() for _ in range(3)]

    n_dev = 3                                          # device staging buffers (no allocator work inside a step)

    def make_e2e_step(layouts, host, run):
        dbufs = [torch.empty(host[0].numel(), dtype=torch.float32, device=dev) for _ in range(n_dev)]
        freed = [torch.cuda.Event() for _ in range(n_dev)]        # the kernels that read the buffer are done
        nxt = [None]                                   # index of the step whose copy was issued ahead

        def issue_h2d(i):
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(freed[i % n_dev])
                dbufs[i % n_dev].copy_(host[i % n_host], non_blocking=True)
                h2d_done[i % n_dev].record(copy_stream)

        def e2e_step(i, prefetch=True):
            # The H2D copy of step i+1 is issued on the copy stream as soon as step i's kernels are queued (what a
            # loader with one sample of look-ahead does); the first step of a region finds nothing prefetched and copies
            # its own inputs, the last one prefetches nothing: a region of n steps contains exactly its own n copies.
            if nxt[0] != i:
                issue_h2d(i)
            stream.wait_event(h2d_done[i % n_dev])
            dbuf = dbufs[i % n_dev]
            d = {k: dbuf[o:o + nel].view(shape) for k, (o, nel, shape) in layouts[i % n_host].items()}
            occ = run(d)
            freed[i % n_dev].record(stream)
            pred_host[i & 1].copy_(occ.reshape(-1), non_blocking=True)
            done[i & 1].record(stream)
            nxt[0] = None
            if prefetch:
                issue_h2d(i + 1)
                nxt[0] = i + 1
            if world > 1:
                pending.append(dist.all_reduce(loss_buf, async_op=True))
            if i > 0:                                  # consume the previous step's prediction on the host
                done[(i - 1) & 1].synchronize()
                consumed[0] += int(pred_host[(i - 1) & 1][0])
        return e2e_step

    def run_e2e(e2e_step):
        for i in range(4):
            e2e_step(i, i < 3)
        steps = max(5, min(K, 100))
        regions = []
        for _ in range(3):                             # three regions of `steps` steps; the median is reported
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            ms_dev = timed_region(steps, lambda i: e2e_step(i, i + 1 < steps))
            wall = time.perf_counter() - t0
            regions.append((max(ms_dev, 0.0) / steps, wall * 1e3 / steps))
        order = sorted(regions)
        return order[1][0], order[1][1], [r[0] for r in regions]

    # (a) the reference-facing call: forward(pts, means, opa, sem, scales, cov) -> logits; arg-max as GaussianHead does
    lay_a, host_a = stage(("pts", "means", "opa", "sem", "scales", "cov"))
    step_a = make_e2e_step(lay_a, host_a, lambda d: module(d["pts"], d["means"], d["opa"], d["sem"], d["scales"], d["cov"]).argmax(dim=1).to(torch.uint8))
    with torch.no_grad():
        e2e_ms, e2e_wall, e2e_regions = run_e2e(step_a)
    h2d = host_a[0].numel() * 4
    d2h = pred_host[0].numel()
    # plain pinned copy of the same bytes on this box: what the PCIe / host path alone costs per step
    with torch.cuda.stream(copy_stream):
        for _ in range(3):
            host_a[0].to(dev, non_blocking=True)
        copy_stream.synchronize()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record(copy_stream)
        for r in range(10):
            host_a[r % n_host].to(dev, non_blocking=True)
        c1.record(copy_stream)
        copy_stream.synchronize()
    h2d_floor_ms = c0.elapsed_time(c1) / 10
    e2e = {"value": world * G_COUNTED / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
           "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms, "wall_ms_per_step": e2e_wall,
           "regions_ms_per_step": e2e_regions, "steps_per_region": max(5, min(K, 100)), "h2d_floor_ms": h2d_floor_ms, "host_numa_binding": numa,
           "api": "local_aggregate.LocalAggregator.forward (drop-in signature, validate=False) + .argmax(1): one pinned "
                  "staging buffer per sample -> H2D on a copy stream (issued one step ahead), forward, arg-max, D2H of the "
                  "uint8 occupancy; host reads prediction i-1 while step i runs; median of three regions of the stated steps"}
    # (b) the grid-resident entry point: only the Gaussians travel (3.5 MB), arg-max fused into the render epilogue
    lay_b, host_b = stage(("means", "opa", "sem", "scales", "cov"))
    pts_grid = module.grid_points(dev)[0]
    step_b = make_e2e_step(lay_b, host_b, lambda d: module.forward_eval(pts_grid, d["means"], d["opa"], d["sem"], d["scales"],
                                                                        d["cov"], layout="nc")["final_occ"])
    with torch.no_grad():
        e2e_b_ms, _, _ = run_e2e(step_b)
    e2e_on_grid = {"value": world * G_COUNTED / (e2e_b_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": host_b[0].numel() * 4,
                   "d2h_bytes_per_step": d2h, "ms_per_step": e2e_b_ms,
                   "api": "LocalAggregator.forward_eval(pts = the grid's resident voxel centres, layout='nc'): logits + fused arg-max"}

    legs = {}
    if not args.no_extras:
        legs = config_legs(dev, world, rank, timed_region, pending, loss_buf, render_alone, peak)
    extras = {}
    if rank == 0 and not args.no_extras:
        extras = side_measurements(dev, kw, inp0, sets[0], desc)

    cpu_baseline = None
    if rank == 0 and world == 1:
        cores = _all_host_threads()
        _cpu_port_once(kw, inp0)
        reps = [_cpu_port_once(kw, inp0) for _ in range(3)]
        sec = sum(reps) / len(reps)
        cpu_baseline = {"value": G_COUNTED / sec, "unit": UNIT, "cores": cores, "kind": "port",
                        "sample": f"3 full forward passes of the {WORKLOAD} sample, {sec:.3f} s each (C/OpenMP oracle)"}
        try:
            # secondary, work-normalised figure (SURVEY.md 8d): in-box (voxel, Gaussian) pairs per second and the fp32
            # rate they stand for at ~56 flop + 1 exp per pair; and the headline sample checked against the CPU port
            pairs = _LAST_PORT["pairs"]
            extras["work"] = {"pairs": pairs, "pairs_per_s": pairs / (render_ms * 1e-3), "flop_per_pair": 56,
                              "fp32_tflops": 56 * pairs / (render_ms * 1e-3) / 1e12,
                              "what": "in-box (voxel, Gaussian) pairs of the sample over the render kernel's time"}
            got = outs[0].float().cpu().numpy()
            want = _LAST_PORT["logits"]
            import numpy as np
            err = np.abs(got - want)
            extras["parity_vs_cpu_port"] = {
                "max_abs_err": float(err.max()), "max_rel_err_above_1e-3": float((err / np.maximum(np.abs(want), 1e-3)).max()),
                "argmax_differences": int((got.argmax(1) != want.argmax(1)).sum()), "voxels": int(got.shape[0]),
                "what": "logits of the timed sample (resident set 0) vs the fp32 C/OpenMP oracle on the host"}
        except Exception as e:
            extras["parity_error"] = repr(e)

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": _config(world, PERTURB),
                "launch": "CUDA graph replay (pack -> list -> render, PDL edges)" if graphs is not None else "3 direct launches per step",
                "clocks": clocks, "e2e": e2e, "e2e_on_grid": e2e_on_grid, "gpu_launches": 3 * K, "roofline": roofline,
                "cpu_baseline": cpu_baseline}
        line.update(legs)
        line.update(extras)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def config_legs(dev, world, rank, timed_region, pending, loss_buf, render_alone, peak):
    """BASELINE.json configs 3, 4 and 5 next to the headline (every rank takes part; rank 0 reports):
    config 3: the 144 000-Gaussian forward, render kernel alone -> roofline_cfg3;
    config 5: forward + backward, 4 samples per GPU in one batched launch per kernel, one scalar all-reduce per step;
    config 4: probabilistic head, 2 samples per GPU (bs 4 over 2 GPUs), forward and backward, HBM and fp32 roofs."""
    import torch
    import torch.distributed as dist
    from gaussianformer_b200 import _lib
    from gaussianformer_b200.splat import LocalAggregator, LocalAggregatorProb, _make_desc, splat_forward_raw
    from gaussianformer_b200.synthetic import make_splat_inputs
    out = {}

    def batch_inputs(name, seeds):
        parts, kws = [], None
        for s in seeds:
            kws, inp, _ = make_splat_inputs(name, seed=s, perturb=False)
            parts.append(inp)
        return kws, {k: torch.cat([p[k] for p in parts], 0).to(dev).contiguous() for k in parts[0]}

    def all_reduce_step():
        if world > 1:
            pending.append(dist.all_reduce(loss_buf, async_op=True))
            if len(pending) > 8:
                pending.pop(0).wait()

    def per_step(n, fn, regions=3):
        """ms per step of a side leg: the median of `regions` timed regions of n steps each (one allocator or host
        hiccup inside a 10-step region would otherwise own the figure)."""
        ms = sorted(timed_region(n, fn) / n for _ in range(regions))
        return ms[len(ms) // 2]

    try:
        # ---- config 3: gs144000 forward, render kernel alone ----
        kw3, t3 = batch_inputs("gs144000", (rank * 100,))
        G3, N3 = t3["means"].shape[1], t3["pts"].shape[1]
        d3 = _make_desc(G3, N3, 18, kw3["H"], kw3["W"], kw3["D"], _lib.GF_SPLAT_BASE, 1, 9, kw3["pc_min"], kw3["grid_size"],
                        float(kw3["scale_multiplier"]), 0, 1, 0)
        cov3 = t3["cov"].reshape(1, G3, 9)

        def call3(i):
            splat_forward_raw(d3, t3["pts"], t3["means"], t3["opa"], t3["sem"], cov3, scales=t3["scales"])
        for i in range(3):
            call3(i)
        k3 = render_alone(call3, 20)
        fwd3 = per_step(20, call3)
        alg3 = _algorithmic_bytes(G3, N3)
        out["roofline_cfg3"] = {"bound": "hbm", "achieved": alg3 / (k3 * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                                "frac": alg3 / (k3 * 1e-3) / 1e9 / peak, "kernel": "render_tile_kernel<18,false>",
                                "kernel_ms": k3, "algorithmic_bytes": alg3, "op_call_ms": fwd3,
                                "workload": "gs144000: 144000 Gaussians -> 200x200x16x18, batch 1"}
        del t3, cov3
    except Exception as e:
        out["roofline_cfg3"] = {"error": repr(e)}

    try:
        # ---- config 5: forward + backward, 4 samples per GPU, one batched launch per kernel ----
        B5 = 4
        kw5, t5 = batch_inputs(WORKLOAD, tuple(rank * 100 + 10 + b for b in range(B5)))
        m5 = LocalAggregator(**kw5).to(dev)
        m5.validate = False
        for k in ("means", "opa", "sem", "cov"):
            t5[k].requires_grad_(True)
        G5, N5 = t5["means"].shape[1], t5["pts"].shape[1]
        up = torch.randn(B5, N5, 18, device=dev)              # resident upstream gradient (dL/dlogits)
        wrt = [t5["means"], t5["opa"], t5["sem"], t5["cov"]]

        def fwd_bwd(i):
            logits = m5(t5["pts"], t5["means"], t5["opa"], t5["sem"], t5["scales"], t5["cov"])
            torch.autograd.grad(logits, wrt, up)
            all_reduce_step()

        def fwd_only(i):
            with torch.no_grad():
                m5(t5["pts"], t5["means"], t5["opa"], t5["sem"], t5["scales"], t5["cov"])
        for i in range(3):
            fwd_bwd(i)
        ms = per_step(20, fwd_bwd)
        ms_f = per_step(20, fwd_only)
        algf, algb = _algorithmic_bytes(G5, N5), _algorithmic_bytes_bwd(G5, N5)
        out["fwd_bwd"] = {"value": world * B5 * G_COUNTED / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms,
                          "fwd_ms": ms_f, "bwd_ms": ms - ms_f, "samples_per_gpu": B5, "global_batch": B5 * world,
                          "hbm_frac_fwd": B5 * algf / (ms_f * 1e-3) / 1e9 / peak,
                          "hbm_frac_bwd": B5 * algb / (max(ms - ms_f, 1e-6) * 1e-3) / 1e9 / peak,
                          "scaling": "weak", "collective": "one scalar all-reduce (NCCL) per step, asynchronous",
                          "what": "BASELINE config 5 (gs25600 bs 32 over 8 GPUs = 4 samples per GPU): module forward + "
                                  "autograd backward, each one batched C-ABI call; max over ranks"}
        del t5, up, m5
    except Exception as e:
        out["fwd_bwd"] = {"error": repr(e)}

    try:
        # ---- config 4: probabilistic head, 2 samples per GPU ----
        B4 = 2
        kw4, t4 = batch_inputs("prob_gs6400", tuple(rank * 100 + 20 + b for b in range(B4)))
        m4 = LocalAggregatorProb(**kw4).to(dev)
        m4.validate = False
        G4, N4 = t4["means"].shape[1], t4["pts"].shape[1]

        def fwd4(i):
            with torch.no_grad():
                m4(t4["pts"], t4["means"], t4["opa"], t4["sem"], t4["scales"], t4["cov"])
            all_reduce_step()
        for i in range(3):
            fwd4(i)
        f_ms = per_step(10, fwd4)
        for k in ("means", "opa", "sem", "cov"):
            t4[k].requires_grad_(True)
        wrt4 = [t4["means"], t4["opa"], t4["sem"], t4["cov"]]
        ups = [torch.randn(B4, N4, 18, device=dev), torch.randn(B4, N4, device=dev), torch.randn(B4, N4, device=dev)]

        def fb4(i):
            lg, bl, de = m4(t4["pts"], t4["means"], t4["opa"], t4["sem"], t4["scales"], t4["cov"])
            torch.autograd.grad([lg, bl, de], wrt4, ups)
            all_reduce_step()
        for i in range(2):
            fb4(i)
        fb_ms = per_step(5, fb4)
        pairs = 1.298e8                                       # in-box pairs per sample of this config (oracle count, seed 0)
        algf, algb = _algorithmic_bytes(G4, N4, prob=True), _algorithmic_bytes_bwd(G4, N4, prob=True)
        b_ms = max(fb_ms - f_ms, 1e-6)
        out["prob"] = {"value": world * B4 * G4 / (f_ms * 1e-3), "unit": UNIT, "fwd_ms": f_ms, "fwd_bwd_ms": fb_ms,
                       "samples_per_gpu": B4, "global_batch": B4 * world,
                       "roofs_fwd": {"hbm_frac": B4 * algf / (f_ms * 1e-3) / 1e9 / peak,
                                     "fp32_tflops": B4 * pairs * 70 / (f_ms * 1e-3) / 1e12,
                                     "fp32_frac": B4 * pairs * 70 / (f_ms * 1e-3) / 1e12 / FP32_PEAK_TFLOPS,
                                     "binding": "fp32 (CUDA cores)"},
                       "roofs_bwd": {"hbm_frac": B4 * algb / (b_ms * 1e-3) / 1e9 / peak,
                                     "fp32_tflops": B4 * pairs * 150 / (b_ms * 1e-3) / 1e12,
                                     "fp32_frac": B4 * pairs * 150 / (b_ms * 1e-3) / 1e12 / FP32_PEAK_TFLOPS,
                                     "binding": "fp32 (CUDA cores) + L1 gather"},
                       "fp32_peak_tflops": FP32_PEAK_TFLOPS, "pairs_per_sample": pairs,
                       "what": "BASELINE config 4 (prob/nuscenes_gs6400, bs 4 over 2 GPUs = 2 samples per GPU): 1.3e8 (voxel, "
                               "Gaussian) pairs per sample at ~70 flop (fwd) / ~150 flop (bwd) each make it compute-bound; "
                               "both roofs reported"}
        del t4, ups, m4
    except Exception as e:
        out["prob"] = {"error": repr(e)}
    torch.cuda.empty_cache()
    return out if rank == 0 else {}


def side_measurements(dev, kw, inp0, resident, desc):
    """Reported next to the headline (not part of it): backward, DAF, and the reference CUDA ops on the same GPU
    when oracle/_ref travelled with the repo."""
    import torch
    from gaussianformer_b200.splat import LocalAggregator
    from gaussianformer_b200.synthetic import make_daf_inputs, make_splat_inputs
    from gaussianformer_b200.ops import DeformableAggregationFunction as DAF
    out = {}

    def timeit(fn, reps=20, warm=3):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize(dev)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize(dev)
        return a.elapsed_time(b) / reps

    try:
        m = LocalAggregator(**kw).to(dev)
        m.validate = False
        t = {k: v.to(dev) for k, v in inp0.items()}
        for k in ("means", "opa", "sem", "cov"):
            t[k].requires_grad_(True)
        logits = m(t["pts"], t["means"], t["opa"], t["sem"], t["scales"], t["cov"])
        g = torch.randn_like(logits)
        out["splat_bwd_ms"] = timeit(lambda: torch.autograd.grad(logits, [t["means"], t["opa"], t["sem"], t["cov"]], g,
                                                                 retain_graph=True), reps=10)
        del logits, g, t
        # BASELINE.json configs[2]: mIoU parity on the 144 000-Gaussian sample (the timing is `roofline_cfg3`)
        kwl, inpl, _ = make_splat_inputs("gs144000", seed=0, perturb=False)
        ml = LocalAggregator(**kwl).to(dev)
        ml.validate = False
        tl = {k: v.to(dev) for k, v in inpl.items()}
        try:
            # north star: mIoU unchanged (SURVEY.md 8d recipe on the 144 000-Gaussian sample, whose arg-max spreads over
            # all 18 classes): fused arg-max of the CUDA path vs the CPU port's arg-max, scored with the reference's MeanIoU
            from gaussianformer_b200.metric import miou_parity, synthetic_labels
            _lg, occ = ml.forward_with_occupancy(tl["pts"], tl["means"], tl["opa"], tl["sem"], tl["scales"], tl["cov"])
            _all_host_threads()
            _cpu_port_once(kwl, inpl)
            want = _LAST_PORT["logits"]
            labels, mask = synthetic_labels(want, want.shape[1])
            r = miou_parity(occ.cpu(), want.argmax(1), labels, mask, want.shape[1])
            out["miou_parity_gs144000"] = {
                "miou_cuda": r["new"][0], "miou_cpu_port": r["ref"][0], "abs_diff": r["abs_diff"],
                "argmax_differences": int((occ.cpu().numpy().astype("int64") != want.argmax(1)).sum()),
                "voxels": int(want.shape[0]),
                "what": "fused arg-max vs the fp32 CPU port; the op-vs-op figure against the reference CUDA op is 0 "
                        "differences (tests/test_parity_full_gpu.py, profiles/r02_parity/)"}
        except Exception as e:
            out["miou_parity_error"] = repr(e)
        del tl
        fms, loc, w = make_daf_inputs(seed=0)
        feat, shape, start = DAF.feature_maps_format([f.to(dev) for f in fms])
        feat = feat.contiguous()
        loc, w = loc.to(dev), w.to(dev)
        dev_maps = [f.to(dev) for f in fms]
        out["daf_format_ms"] = timeit(lambda: DAF.feature_maps_format(dev_maps)[0], reps=10)

        def torch_format():      # the reference's route: reshape + cat + permute, then the copy .contiguous() makes
            bs, cams, ch = dev_maps[0].shape[:3]
            return torch.cat([m.reshape(bs, cams, ch, -1) for m in dev_maps], dim=-1).permute(0, 1, 3, 2).contiguous()
        out["ref_format_torch_ms"] = timeit(torch_format, reps=10)
        del dev_maps
        out["daf_fwd_ms"] = timeit(lambda: DAF.apply(feat, shape, start, loc, w), reps=10)
        out["daf_fwd_alg_gbs"] = 4 * (feat.numel() + loc.numel() + w.numel() + loc.shape[1] * 128) / (out["daf_fwd_ms"] * 1e-3) / 1e9
    except Exception as e:  # side figures must never sink the headline
        out["extras_error"] = repr(e)
    try:
        # fused caller path (SURVEY.md 8f-2): masked softmax + op + key-point sum, against the same three steps done
        # the reference's way (PyTorch softmax -> our drop-in op -> .sum) on the same inputs
        from gaussianformer_b200.ops import deformable_aggregation_fused
        from gaussianformer_b200.synthetic import make_daf_fused_inputs, reference_fused_composition
        fms, loc, lg, pm, _ = make_daf_fused_inputs(seed=0)
        feat, shape, start = DAF.feature_maps_format([f.to(dev) for f in fms])
        feat = feat.contiguous()
        loc, lg, pm = loc.to(dev), lg.to(dev), pm.to(dev)
        with torch.no_grad():
            out["daf_fused_fwd_ms"] = timeit(lambda: deformable_aggregation_fused(feat, shape, start, loc, lg, pm), reps=10)
            out["daf_unfused_fwd_ms"] = timeit(lambda: reference_fused_composition(DAF.apply, feat, shape, start, loc, lg, pm), reps=10)
        feat.requires_grad_(True); loc.requires_grad_(True); lg.requires_grad_(True)
        g = torch.randn(1, lg.shape[1], feat.shape[-1], device=dev)

        def fwd_bwd(fn):
            o = fn(feat, shape, start, loc, lg, pm)
            return torch.autograd.grad(o, [feat, loc, lg], g)
        out["daf_fused_fwd_bwd_ms"] = timeit(lambda: fwd_bwd(deformable_aggregation_fused), reps=5)
        out["daf_unfused_fwd_bwd_ms"] = timeit(lambda: fwd_bwd(lambda *a: reference_fused_composition(DAF.apply, *a)), reps=5)
        del feat, loc, lg, pm, g
    except Exception as e:
        out["daf_fused_error"] = repr(e)
    try:
        # the reference's own fallback for the sampling op (PyTorch grid_sample route, deformable_module.py:307-353,
        # restated in oracle.daf_torch_fallback) on the host cores, on a bounded sample of the same workload
        import oracle
        fms, loc, w = make_daf_inputs(seed=0)
        nsub = 23040                                        # one tenth of the 230 400 sampling points
        loc_s, w_s = loc[:, :nsub].contiguous(), w[:, :nsub].contiguous()
        with torch.no_grad():
            oracle.daf_torch_fallback(fms, loc_s, w_s, 4)
            t0 = time.perf_counter()
            oracle.daf_torch_fallback(fms, loc_s, w_s, 4)
            sec = time.perf_counter() - t0
        out["daf_cpu_fallback"] = {"ms_per_full_call_extrapolated": sec * 1e3 * loc.shape[1] / nsub, "sample_ms": sec * 1e3,
                                   "sample": f"{nsub} of {loc.shape[1]} sampling points, 6 cameras x 4 levels, C = 128",
                                   "cores": torch.get_num_threads(), "kind": "port",
                                   "what": "reference's PyTorch fallback of the op (grid_sample + weighted fusion) on the host"}
    except Exception as e:
        out["daf_cpu_fallback"] = {"error": repr(e)}
    try:
        from oracle import build_ref
        if build_ref.available("gf_ref_daf"):
            mod = build_ref.load_ref("gf_ref_daf")
            fms, loc, w = make_daf_inputs(seed=0)
            feat, shape, start = DAF.feature_maps_format([f.to(dev) for f in fms])
            feat = feat.contiguous()
            loc, w, shape_i, start_i = loc.to(dev), w.to(dev), shape.int(), start.int()
            ref_f = timeit(lambda: mod.deformable_aggregation_forward(feat, shape_i, start_i, loc, w), reps=10)
            g = torch.randn(1, loc.shape[1], 128, device=dev)
            gf, gl, gw = torch.zeros_like(feat), torch.zeros_like(loc), torch.zeros_like(w)
            ref_b = timeit(lambda: mod.deformable_aggregation_backward(feat, shape_i, start_i, loc, w, g, gf, gl, gw), reps=5)
            feat.requires_grad_(True); loc.requires_grad_(True); w.requires_grad_(True)
            o = DAF.apply(feat, shape, start, loc, w)
            out["daf_bwd_ms"] = timeit(lambda: torch.autograd.grad(o, [feat, loc, w], g, retain_graph=True), reps=5)
            out["ref_daf_op"] = {"fwd_ms": ref_f, "bwd_kernel_ms": ref_b, "what": "reference deformable_aggregation op "
                                 "compiled for sm_100a, same GPU, same inputs (backward without its three zero fills)"}
    except Exception as e:
        out["ref_daf_op"] = {"error": repr(e)}
    try:
        from oracle import build_ref
        if build_ref.available("gf_ref_localagg"):
            mod = build_ref.load_ref("gf_ref_localagg")
            t = {k: v[0].to(dev) for k, v in inp0.items()}
            pc_min = torch.tensor(kw["pc_min"], device=dev)[None]

            def ref_call():   # the reference's Python wrapper + native op (asserts included)
                pi = ((t["pts"] - pc_min) / kw["grid_size"]).to(torch.int)
                assert pi.min() >= 0
                mi = ((t["means"] - pc_min) / kw["grid_size"]).to(torch.int)
                assert mi.min() >= 0
                radii = torch.ceil(t["scales"].max(dim=-1)[0] * kw["scale_multiplier"] / kw["grid_size"]).to(torch.int)
                assert radii.min() >= 1
                cov6 = t["cov"].flatten(1)[:, [0, 4, 8, 1, 5, 2]]
                return mod.local_aggregate(t["pts"], pi, t["means"], mi, t["opa"], t["sem"], radii, cov6,
                                           kw["H"], kw["W"], kw["D"])
            ref_fwd = timeit(ref_call, reps=10)
            R, logits, geom, binning, img = ref_call()
            pi = ((t["pts"] - pc_min) / kw["grid_size"]).to(torch.int)
            cov6 = t["cov"].flatten(1)[:, [0, 4, 8, 1, 5, 2]].contiguous()
            g = torch.randn_like(logits)
            ref_bwd = timeit(lambda: mod.local_aggregate_backward(geom, binning, img, kw["H"], kw["W"], kw["D"], R,
                                                                  t["means"], t["pts"], pi, cov6, t["opa"], t["sem"], g),
                             reps=3, warm=1)
            out["ref_cuda_op"] = {"fwd_ms": ref_fwd, "bwd_ms": ref_bwd, "what": "reference localagg op "
                                  "(its Python prep + sort-based kernels; backward = native call only) compiled for "
                                  "sm_100a, same GPU, same sample"}
    except Exception as e:
        out["ref_cuda_op"] = {"error": repr(e)}
    return out


if __name__ == "__main__":
    main()

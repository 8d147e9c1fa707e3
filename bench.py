#!/usr/bin/env python
"""bench.py — DIB-R fwd+bwd throughput on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W          # this repo's kernels
    python bench.py --impl reference --gpus N ...          # reference arm (CPU path)

Workload (`config.workload` = "c4_shard"): the per-GPU shard of BASELINE.json
configs[3] — 32 views per GPU of a ~20k-face mesh (icosphere level 5 = 20480
faces, jittered, random rotation and camera; SURVEY.md §8d generator G1) at
1024x1024, D = 3 feature channels, fp32.  One "step" = dibr_rasterization forward
+ backward (grads wrt face_vertices_image and face_features) over the shard;
with N > 1 every rank renders its own 32 views (weak scaling) and the per-view
gradients are all-gathered (--gather: stores into peer memory over NVLink when
the box offers symmetric memory, else NCCL).  Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "DIB-R fwd+bwd Mpixels/sec at 1024^2 per GPU; achieved HBM GB/s vs peak"
UNIT = "Mpixels/s"
WORKLOADS = {
    # name: (views per GPU, icosphere level, H, W, D, radial vertex jitter)
    "c4_shard": (32, 5, 1024, 1024, 3, 0.05),
    "c2": (8, 4, 256, 256, 3, 0.05),
    "c3": (64, 5, 512, 512, 3, 0.05),
    # configs[4]: one 1.3 M-triangle mesh, 8 views.  "c5" scales the jitter with the edge
    # length (a bumpy surface, ~3 px^2 triangles); "c5_spiky" keeps the level-5 jitter,
    # 8x the edge length: sliver triangles with 20-px boxes, >2000 soft-mask candidates per
    # tile (the index-windowed path) - a stress case, not a mesh anyone renders.
    "c5": (8, 8, 2048, 2048, 3, 0.05 / 8),
    "c5_spiky": (8, 8, 2048, 2048, 3, 0.05),
    "tiny": (2, 3, 128, 128, 3, 0.05),
}
SIGMAINV, BOXLEN, KNUM, MULT, EPS = 7000.0, 0.02, 30, 1000.0, 1e-8


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=20)
    p.add_argument("--warmup", type=int, default=5)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--workload", default="c4_shard", choices=list(WORKLOADS))
    p.add_argument("--cpu-seconds", type=float, default=20.0,
                   help="CPU work budget for the cpu_baseline sample")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-ref-cuda", action="store_true")
    p.add_argument("--no-e2e-images", action="store_true")
    p.add_argument("--e2e-graph", action="store_true",
                   help="N = 1: also time the public API's CUDA-graph fast path (make_graphed_dibr_rasterization)")
    p.add_argument("--ref-cuda-views", type=int, default=2)
    p.add_argument("--features", default="fp32", choices=["fp32", "bf16"],
                   help="storage of face_features / features / grad_features (arithmetic is fp32 either "
                        "way); BASELINE configs[3] names bf16, the reference itself only has fp32/fp64")
    p.add_argument("--cache-fraction", type=float, default=None,
                   help="override kaolin_b200.render.mesh._host.CACHE_TILE_FRACTION (share of the screen tiles "
                        "whose soft-mask hits may be cached for backward)")
    p.add_argument("--graph", action="store_true",
                   help="N = 1: capture the resident forward+backward step in a CUDA graph and time replays "
                        "(what launch-bound sizes such as c2 gain from it)")
    p.add_argument("--bwd-chunks", type=int, default=None,
                   help="N > 1: view chunks of the BACKWARD (dibr_b200_backward_views); chunk i's gradient all-gathers "
                        "travel while chunk i+1 computes. Default 1 (the feature gradient's gather overlaps the "
                        "soft-mask branch): measured at N = 2, two chunks cost +0.15 ms of backward compute "
                        "(half-size launches) for at most 0.1 ms of hidden exchange at N = 8")
    p.add_argument("--gather", default="auto", choices=["auto", "nccl", "peer", "peer_sm", "peer_mc"],
                   help="N > 1: transport of the gradient all-gather. peer = stores into the peers' memory over "
                        "NVLink by the copy engines (kaolin_b200.multi_gpu.PeerGradAllGather), peer_sm = the same by "
                        "the dibr_b200_peer_push kernel, nccl = all_gather_into_tensor; auto = peer when CUDA "
                        "symmetric memory can be set up on this box, else nccl")
    p.add_argument("--push-ctas", type=int, default=32, help="--gather peer_sm: grid of the push kernel")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="after the timed steps, write what the last timed step computed (features, soft_mask, "
                        "face_idx, grad_face_vertices_image, grad_face_features) as DIR/<name>.npy in float32 / "
                        "float64, at most 64 MB in all (a fixed seeded sample of the pixels / faces when larger). "
                        "--impl ours only. With --gpus N, rank 0 writes: the images of its own views and the "
                        "gradients as every rank receives them, all-gathered over the N x views")
    p.add_argument("--chunks", type=int, default=1,
                   help="N > 1: 1 = the all-gather of grad_face_features overlaps the soft-mask branch of "
                        "the backward (default); k > 1 = k view-chunks per step, chunk i's all-gather "
                        "overlaps chunk i+1 (measured slower at 32 views per GPU: smaller launches)")
    args = p.parse_args()
    if args.dump_outputs and args.impl != "ours":
        p.error("--dump-outputs writes what the timed GPU step computed: --impl ours only")
    return args


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            d = json.load(open(path))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def algorithmic_bytes(B, F, H, W, D, s=4):
    """SURVEY.md §8(d): compulsory HBM traffic of the fused path (fp32: s = 4)."""
    P = B * H * W
    fwd = P * (D * s + 4 + 8 + 12) + B * F * (12 + 24 + 3 * D * s)
    bwd = P * (D * s + 4 + 8 + 12) + B * F * (48 + 6 * D * s)
    bwd_raster = P * (D * s + 8 + 12) + B * F * (24 + 3 * D * s + 24 + 3 * D * s)
    return {"fwd": fwd, "bwd": bwd, "total": fwd + bwd, "bwd_raster": bwd_raster}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "20", "-i", str(index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL,
                text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for n, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def effective_cores():
    """Host threads the CPU arm may really use: min(CPUs this process may run on, cgroup CPU
    quota).  torchrun exports OMP_NUM_THREADS=1 (ignored on purpose); a container with a CFS
    quota of q CPUs but 128 visible ones makes a 128-thread OpenMP team 10x SLOWER than q
    threads (round 1: 0.016 vs 0.21 Mpx/s for the same commit), so the quota is honoured."""
    try:
        affinity = len(os.sched_getaffinity(0))
    except AttributeError:
        affinity = os.cpu_count() or 1
    quota = None
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:           # cgroup v2: "<quota|max> <period>"
            q, per = f.read().split()
            if q != "max":
                quota = float(q) / float(per)
    except Exception:
        try:                                                  # cgroup v1
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            quota = None
    used = affinity if quota is None else max(1, min(affinity, int(quota + 0.5)))
    return used, {"affinity": affinity, "cgroup_quota_cpus": quota, "used": used}


def make_scene(workload, rank):
    from kaolin_b200 import synthetic
    B, level, H, W, D, jitter = WORKLOADS[workload]
    fvz, fvi, fnz = synthetic.icosphere_views(B, level, seed=1234 + 17 * rank, jitter=jitter,
                                              same_mesh=(level >= 8))
    ff = synthetic.random_features(B, fvz.shape[1], D, seed=99 + rank)
    return B, fvz.shape[1], H, W, D, fvz, fvi, fnz, ff


# ---------------------------------------------------------------------------
def cpu_sample(workload, budget_s, threads=None):
    """Oracle (CPU restatement of the reference kernels) on a bounded sample:
    a centred strip of rows of ONE view of the workload, all host threads."""
    import oracle
    oracle.build()
    B, F, H, W, D, fvz, fvi, fnz, ff = make_scene(workload, 0)
    fvz, fvi, fnz, ff = fvz[:1], fvi[:1], fnz[:1], ff[:1]
    rng = np.random.default_rng(0)
    g_feat = rng.uniform(size=(1, H, W, D)).astype(np.float32)
    g_soft = rng.uniform(size=(1, H, W)).astype(np.float32)
    if not threads:
        threads, cores_info = effective_cores()
    else:
        cores_info = {"used": threads}
    oracle.set_threads(threads)
    cores = threads

    def strips_for(nblocks, rows_per_block=4):
        nblocks = max(1, min(H // rows_per_block, nblocks))
        pitch = H / nblocks                      # blocks spread evenly over the image height
        return [(int(i * pitch), int(i * pitch) + rows_per_block) for i in range(nblocks)]

    probe = strips_for(4)
    s = oracle.RowSample(H, W, fvz, fvi, ff, fnz, g_feat, g_soft, 0, 0, SIGMAINV, BOXLEN, KNUM, MULT, EPS,
                         strips=probe)
    s.run()                                       # touch pages, start the OpenMP team
    t = time.perf_counter(); s.run(); dt = time.perf_counter() - t
    # 1 thread vs the full team on the same 16 rows: a starved arm (quota, noisy neighbours) shows
    # up as a speed-up far below the thread count
    if threads > 1:
        oracle.set_threads(1)
        t = time.perf_counter(); s.run(); dt1 = time.perf_counter() - t
        oracle.set_threads(threads)
        cores_info = dict(cores_info, scaling_probe={"rows": 16, "threads_1_s": dt1, f"threads_{threads}_s": dt,
                                                     "speedup": dt1 / max(dt, 1e-9)})
    nblocks = int(max(4, len(probe) * budget_s / max(dt, 1e-6)))
    strips = strips_for(nblocks)
    s = oracle.RowSample(H, W, fvz, fvi, ff, fnz, g_feat, g_soft, 0, 0, SIGMAINV, BOXLEN, KNUM, MULT, EPS,
                         strips=strips)
    rows = sum(b - a for a, b in strips)
    cpu_sample.cores_info = cores_info
    return s, cores, (f"{rows} of {H} rows ({len(strips)} evenly spaced 4-row blocks) of 1 view of "
                      f"{workload} ({W}x{H}, {F} faces)")


def run_reference(args):
    """Reference arm: the reference has no CPU implementation of this path
    (rasterization.cpp:95-102 raises without CUDA), so this times the oracle port
    (kind "port") on the host cores; rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    per_step = max(0.5, min(20.0, 120.0 / max(1, args.steps + args.warmup)))
    s, cores, desc = cpu_sample(args.workload, per_step)
    for _ in range(args.warmup):
        s.run()
    t = time.perf_counter()
    for _ in range(args.steps):
        s.run()
    dt = (time.perf_counter() - t) / max(1, args.steps)
    val = s.pixels / dt / 1e6
    B, level, H, W, D, _ = WORKLOADS[args.workload]
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": args.workload, "vertex_jitter": WORKLOADS[args.workload][5],
                   "views_per_gpu": B, "faces_per_view": 20 * 4 ** level,
                   "height": H, "width": W, "feat_dim": D, "knum": KNUM, "sample": desc},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": desc,
                         "cores_detail": getattr(cpu_sample, "cores_info", None)},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from kaolin_b200 import _lib
    from kaolin_b200.render.mesh import _host, dibr_rasterization
    from kaolin_b200.multi_gpu import (ChunkedGradAllGather, PipelinedGradAllGather, chunk_ranges,
                                       make_grad_all_gather, pipelined_backward_all_gather)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py (impl=ours) needs a CUDA device; there is no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # one box, NVLink only (north_star): no IB / socket transports; the collective kernels run
        # on a HIGH-PRIORITY stream so that they get SM slots as soon as any CTA retires instead of
        # queueing behind the (tens of thousands of CTAs of the) next kernels of the step
        os.environ.setdefault("NCCL_P2P_LEVEL", "NVL")
        os.environ.setdefault("NCCL_IB_DISABLE", "1")
        os.environ.setdefault("NCCL_NET_DISABLE", "1")
        opts = None
        try:
            opts = dist.ProcessGroupNCCL.Options(is_high_priority_stream=True)
        except Exception:
            opts = None
        dist.init_process_group("nccl", device_id=dev, pg_options=opts)
    _lib.lib()
    if args.cache_fraction is not None:
        _host.CACHE_TILE_FRACTION = float(args.cache_fraction)

    B, F, H, W, D, fvz, fvi, fnz, ff = make_scene(args.workload, rank)
    pin = lambda a: torch.from_numpy(a).pin_memory()
    fdt = torch.bfloat16 if args.features == "bf16" else torch.float32
    h_fvz, h_fvi, h_fnz = pin(fvz), pin(fvi), pin(fnz)
    h_ff = torch.from_numpy(ff).to(fdt).pin_memory()
    d_fvz, d_fvi, d_fnz, d_ff = (t.to(dev) for t in (h_fvz, h_fvi, h_fnz, h_ff))
    gen = torch.Generator(device=dev); gen.manual_seed(4321 + rank)
    g_feat = torch.rand((B, H, W, D), device=dev, generator=gen).to(fdt)
    g_soft = torch.rand((B, H, W), device=dev, generator=gen)
    boxlen_m = BOXLEN * MULT
    mode = _lib.RASTER | _lib.SOFT_MASK

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- resident path: C ABI with device pointers (value) ----------------
    # N > 1: the all-gather of grad_face_features (final after the rasterize branch of the
    # backward) travels while the soft-mask branch runs; grad_face_vertices_image follows.
    spans = chunk_ranges(B, args.chunks) if world > 1 else [(0, B)]
    bwd_chunks = args.bwd_chunks if args.bwd_chunks is not None else 1
    pipelined = world > 1 and len(spans) == 1 and bwd_chunks > 1

    # transport of the exchange, decided once (collectively) before the warm-up
    transport = {"used": None}

    def new_gather():
        g, used = make_grad_all_gather(B * world, (B, F, 3, 2), (B, F, 3, D), dev,
                                       transport=transport["used"] or args.gather, ctas=args.push_ctas)
        transport["used"] = used
        return g

    if world > 1 and len(spans) == 1 and not pipelined:
        new_gather()
        if rank == 0:
            print(f"[bench] gradient all-gather transport: {transport['used']}", file=sys.stderr)

    def step_resident(ev=None):
        chunked = ChunkedGradAllGather(B) if world > 1 and len(spans) > 1 else None
        images = []
        for ci, (c0, c1) in enumerate(spans):
            if ev: ev[3 * ci].record()
            feat, idx, wts, soft, ws = _host.forward(mode, H, W, d_fvz[c0:c1], d_fvi[c0:c1], d_ff[c0:c1],
                                                     d_fnz[c0:c1], None, MULT, EPS, SIGMAINV, boxlen_m, KNUM)
            images.append((feat, soft, idx))
            if ev: ev[3 * ci + 1].record()
            bwd = lambda hook=None: _host.backward(H, W, g_feat[c0:c1], g_soft[c0:c1], idx, wts, soft,
                                                   d_fvi[c0:c1], d_ff[c0:c1], MULT, EPS, SIGMAINV, boxlen_m,
                                                   KNUM, ws, True, feature_grad_hook=hook)
            if pipelined:
                l_fvi = torch.empty_like(d_fvi)
                l_ff = torch.empty(d_ff.shape, dtype=torch.float32, device=dev)
                run = lambda v0, v1, hook: _host.backward(H, W, g_feat, g_soft, idx, wts, soft, d_fvi, d_ff, MULT, EPS,
                                                          SIGMAINV, boxlen_m, KNUM, ws, True, feature_grad_hook=hook,
                                                          views=(v0, v1), out=(l_fvi, l_ff))
                g_fvi, g_ff = pipelined_backward_all_gather(B, bwd_chunks, run, l_fvi, l_ff)
                if ev: ev[3 * ci + 2].record()
            elif world > 1 and chunked is None:
                gather = new_gather()
                g_fvi, g_ff = bwd(gather.hook)
                if ev: ev[3 * ci + 2].record()
                g_fvi, g_ff = gather.finish(g_fvi)
            else:
                g_fvi, g_ff = bwd()
                if ev: ev[3 * ci + 2].record()
                if chunked is not None:
                    chunked.submit(c0, c1, [g_fvi, g_ff])
        if chunked is not None:
            g_fvi, g_ff = chunked.finish()
        return images, g_fvi, g_ff

    graph = None
    if args.graph and world == 1:
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            step_resident()
        torch.cuda.current_stream(dev).wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            graph_out = step_resident()
        eager_step = step_resident

        def step_resident(ev=None):     # noqa: F811 - replay; per-phase events do not exist inside a graph
            if ev: ev[0].record()
            graph.replay()
            if ev: ev[1].record(); ev[2].record()
            return graph_out

    for _ in range(args.warmup):
        step_resident()
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(3 * len(spans))] for _ in range(args.steps)]
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # clocks are sampled on rank 0 only (8 nvidia-smi pollers at 20 ms inside a 100 ms window were one
    # suspect for round 1's slow N = 8 number) and the poller is spawned BEFORE the barrier: spawning it
    # after made rank 0 enter the timed loop milliseconds late, and every other rank's first all-gather
    # waited for it (one 3.5 ms step per rank in the first N = 8 run of this round)
    sampler = ClockSampler(torch.cuda.current_device() if "CUDA_VISIBLE_DEVICES" not in os.environ else local) \
        if rank == 0 else None
    barrier()
    start.record()
    for k in range(args.steps):
        last = step_resident(evs[k])
        if k + 1 < args.steps:
            del last                    # each step's outputs are released before the next step, as in a loop
    end.record()
    barrier()
    clocks = sampler.stop() if sampler is not None else None
    total_ms = start.elapsed_time(end)
    # per-step device time on this rank (event at the start of step k -> start of step k+1)
    marks = [e[0] for e in evs] + [end]
    step_ms = [marks[k].elapsed_time(marks[k + 1]) for k in range(args.steps)]
    nch = len(spans)
    fwd_ms = statistics.mean(sum(e[3 * c].elapsed_time(e[3 * c + 1]) for c in range(nch)) for e in evs)
    bwd_ms = statistics.mean(sum(e[3 * c + 1].elapsed_time(e[3 * c + 2]) for c in range(nch)) for e in evs)
    t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
    per_rank = None
    if world > 1:
        mine = torch.tensor([total_ms / args.steps, min(step_ms), statistics.median(step_ms), max(step_ms)],
                            device=dev, dtype=torch.float64)
        allr = torch.empty((world, 4), device=dev, dtype=torch.float64)
        dist.all_gather_into_tensor(allr, mine)
        per_rank = [[round(float(x), 4) for x in row] for row in allr.cpu()]
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_per_step = float(t.item()) / args.steps
    value = world * B * H * W / (ms_per_step * 1e-3) / 1e6
    step_stats = {"min": min(step_ms), "median": statistics.median(step_ms), "max": max(step_ms),
                  "rank": 0, "per_rank_mean_min_median_max": per_rank}
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)
    del last

    # ---- the backward scatter kernel alone (roofline kernel) ---------------
    feat, idx, wts, soft, ws = _host.forward(mode, H, W, d_fvz, d_fvi, d_ff, d_fnz, None, MULT, EPS,
                                             SIGMAINV, boxlen_m, KNUM)
    covered = float((idx >= 0).float().mean().item())
    rb = [torch.cuda.Event(enable_timing=True) for _ in range(2 * args.steps)]
    for _ in range(2):
        _host.backward(H, W, g_feat, None, idx, wts, None, d_fvi, d_ff, MULT, EPS, 0., 0., 0, None, False)
    torch.cuda.synchronize()
    for k in range(args.steps):
        rb[2 * k].record()
        _host.backward(H, W, g_feat, None, idx, wts, None, d_fvi, d_ff, MULT, EPS, 0., 0., 0, None, False)
        rb[2 * k + 1].record()
    torch.cuda.synchronize()
    raster_bwd_ms = statistics.mean(rb[2 * k].elapsed_time(rb[2 * k + 1]) for k in range(args.steps))
    band_px = int(((idx < 0) & (soft > 0)).sum().item())     # uncovered pixels with a soft-mask value
    del feat, idx, wts, soft, ws

    # ---- every kernel of the step, CUDA events around each launch (library trace) ----------
    kernel_ms = {}
    kernel_order = []
    tsteps = max(3, min(10, args.steps))
    for _ in range(tsteps):
        _lib.trace_begin()
        f_, i_, w_, s_, ws_ = _host.forward(mode, H, W, d_fvz, d_fvi, d_ff, d_fnz, None, MULT, EPS, SIGMAINV,
                                            boxlen_m, KNUM)
        _host.backward(H, W, g_feat, g_soft, i_, w_, s_, d_fvi, d_ff, MULT, EPS, SIGMAINV, boxlen_m, KNUM, ws_, True)
        for name, ms in _lib.trace_end():
            if name not in kernel_ms:
                kernel_ms[name] = []
                kernel_order.append(name)
            kernel_ms[name].append(ms)
        del f_, i_, w_, s_, ws_

    # ---- e2e: public API, host buffers, H2D + D2H inside the timed region --
    # Every step copies ITS inputs from pinned host memory and returns ITS gradients
    # (+ a scalar) to pinned host memory.  As any training loop would, the copies run
    # on their own streams so that step i+1's upload and step i-1's download overlap
    # step i's kernels (double-buffered device inputs / host outputs); the host reads
    # every step's result (one step behind) before the timed region ends.
    NB = 2
    s_h2d, s_d2h = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    s_cmp = torch.cuda.current_stream(dev)
    dev_in = []
    for _ in range(NB):
        bufs = [torch.empty_like(x, device=dev) for x in (h_fvz, h_fvi, h_ff, h_fnz)]
        bufs[1].requires_grad_(True); bufs[2].requires_grad_(True)
        dev_in.append(bufs)
    host_out = [(torch.empty((B, F, 3, 2), dtype=torch.float32).pin_memory(),
                 torch.empty((B, F, 3, D), dtype=fdt).pin_memory(),
                 torch.empty((1,), dtype=torch.float32).pin_memory()) for _ in range(NB)]
    dev_out = [tuple(torch.empty(t.shape, dtype=t.dtype, device=dev) for t in host_out[k]) for k in range(NB)]
    ev_free = [None] * NB      # device inputs of slot consumed by compute
    ev_read = [None] * NB      # host outputs of slot downloaded
    state = {"i": 0, "checksum": 0.0}

    def step_e2e():
        i = state["i"]; slot = i % NB
        a_fvz, a_fvi, a_ff, a_fnz = dev_in[slot]
        with torch.cuda.stream(s_h2d):
            if ev_free[slot] is not None:
                s_h2d.wait_event(ev_free[slot])
            with torch.no_grad():
                a_fvz.copy_(h_fvz, non_blocking=True); a_fvi.copy_(h_fvi, non_blocking=True)
                a_ff.copy_(h_ff, non_blocking=True); a_fnz.copy_(h_fnz, non_blocking=True)
            ev_up = torch.cuda.Event(); ev_up.record(s_h2d)
        s_cmp.wait_event(ev_up)
        if world == 1:
            a_fvi.grad = None; a_ff.grad = None
            feat, soft, idx = dibr_rasterization(H, W, a_fvz, a_fvi, a_ff, a_fnz, SIGMAINV, BOXLEN, KNUM)
            torch.autograd.backward([feat, soft], [g_feat, g_soft])
            g1, g2 = a_fvi.grad, a_ff.grad
            loss = (soft.detach().sum() / soft.numel()).reshape(1)
        elif len(spans) == 1:
            a_fvi.grad = None; a_ff.grad = None
            feat, soft, idx = dibr_rasterization(H, W, a_fvz, a_fvi, a_ff, a_fnz, SIGMAINV, BOXLEN, KNUM)
            if pipelined:
                gather = PipelinedGradAllGather(chunks=bwd_chunks).attach(soft)
                torch.autograd.backward([feat, soft], [g_feat, g_soft])
                full = gather.finish()
            else:
                gather = new_gather().attach(soft)
                torch.autograd.backward([feat, soft], [g_feat, g_soft])
                full = gather.finish(a_fvi.grad, a_ff.grad)
            g1, g2 = full[0][rank * B:(rank + 1) * B], full[1][rank * B:(rank + 1) * B]
            loss = (soft.detach().sum() / soft.numel()).reshape(1)
        else:
            gather = ChunkedGradAllGather(B)
            loss = torch.zeros(1, device=dev)
            for c0, c1 in spans:
                c_fvi = a_fvi[c0:c1].detach().requires_grad_(True)
                c_ff = a_ff[c0:c1].detach().requires_grad_(True)
                feat, soft, idx = dibr_rasterization(H, W, a_fvz[c0:c1], c_fvi, c_ff, a_fnz[c0:c1],
                                                     SIGMAINV, BOXLEN, KNUM)
                torch.autograd.backward([feat, soft], [g_feat[c0:c1], g_soft[c0:c1]])
                gather.submit(c0, c1, [c_fvi.grad, c_ff.grad])
                loss += soft.detach().sum() / (B * H * W)
            full = gather.finish()
            g1, g2 = full[0][rank * B:(rank + 1) * B], full[1][rank * B:(rank + 1) * B]
        if ev_read[slot] is not None:          # host has consumed this slot's previous result
            ev_read[slot].synchronize()
            state["checksum"] += float(host_out[slot][2][0])
        # results go to a per-slot device staging buffer on the compute stream (39 MB, ~12 us),
        # so no autograd/allocator-owned tensor is ever touched by the download stream
        # (record_stream would delay the reuse of their blocks and make the caching
        # allocator fall back to cudaMalloc now and then: sporadic 2x slow steps)
        st_fvi, st_ff, st_loss = dev_out[slot]
        with torch.no_grad():
            st_fvi.copy_(g1); st_ff.copy_(g2); st_loss.copy_(loss)
        ev_done = torch.cuda.Event(); ev_done.record(s_cmp)
        ev_free[slot] = ev_done
        with torch.cuda.stream(s_d2h):
            s_d2h.wait_event(ev_done)
            host_out[slot][0].copy_(st_fvi, non_blocking=True)
            host_out[slot][1].copy_(st_ff, non_blocking=True)
            host_out[slot][2].copy_(st_loss, non_blocking=True)
            # blocking=True: the host SLEEPS in ev_read.synchronize() instead of spinning - with one process per
            # GPU under a CPU quota (8 ranks on a 16-CPU cgroup) eight spinning waiters starve the autograd threads
            ev = torch.cuda.Event(blocking=True); ev.record(s_d2h)
        ev_read[slot] = ev
        state["i"] = i + 1

    def drain():
        for slot in range(NB):
            if ev_read[slot] is not None:
                ev_read[slot].synchronize()
                state["checksum"] += float(host_out[slot][2][0])
                ev_read[slot] = None
        torch.cuda.synchronize()

    for _ in range(max(3, args.warmup)):
        step_e2e()
    drain()
    barrier()
    t0 = time.perf_counter()
    start.record()
    for _ in range(args.steps):
        step_e2e()
    drain()                                      # every step's result has reached the host
    end.record()
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    t = torch.tensor([max(start.elapsed_time(end), 0.0)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = float(t.item()) / args.steps
    e2e_value = world * B * H * W / (e2e_ms * 1e-3) / 1e6
    h2d = sum(x.numel() * x.element_size() for x in (h_fvz, h_fvi, h_fnz, h_ff))
    d2h = sum(x.numel() * x.element_size() for x in host_out[0])

    # ---- e2e_images (N = 1): as e2e, but the drop-in API's RETURN VALUES (features, soft_mask,
    # face_idx) are downloaded as well - what a caller that post-processes the images on the
    # host pays; PCIe-bound (28+ B per pixel)
    e2e_images = None
    if world == 1 and not args.no_e2e_images:
        n_img = 3
        h_img = (torch.empty((B, H, W, D), dtype=fdt).pin_memory(), torch.empty((B, H, W), dtype=torch.float32).pin_memory(),
                 torch.empty((B, H, W), dtype=torch.int64).pin_memory())
        def step_images():
            a_fvz, a_fvi, a_ff, a_fnz = dev_in[0]
            with torch.no_grad():
                a_fvz.copy_(h_fvz, non_blocking=True); a_fvi.copy_(h_fvi, non_blocking=True)
                a_ff.copy_(h_ff, non_blocking=True); a_fnz.copy_(h_fnz, non_blocking=True)
            a_fvi.grad = None; a_ff.grad = None
            feat, soft, idx = dibr_rasterization(H, W, a_fvz, a_fvi, a_ff, a_fnz, SIGMAINV, BOXLEN, KNUM)
            torch.autograd.backward([feat, soft], [g_feat, g_soft])
            h_img[0].copy_(feat.detach(), non_blocking=True); h_img[1].copy_(soft.detach(), non_blocking=True)
            h_img[2].copy_(idx, non_blocking=True)
            host_out[0][0].copy_(a_fvi.grad, non_blocking=True); host_out[0][1].copy_(a_ff.grad, non_blocking=True)
        step_images(); torch.cuda.synchronize()
        start.record()
        for _ in range(n_img):
            step_images()
        end.record(); torch.cuda.synchronize()
        ims = start.elapsed_time(end) / n_img
        e2e_images = {"value": B * H * W / (ims * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": ims, "steps": n_img,
                      "d2h_bytes_per_step": d2h + sum(x.numel() * x.element_size() for x in h_img)}
        del h_img

    # ---- e2e through the CUDA-graph fast path of the public API (launch-bound sizes) --------
    e2e_graphed = None
    if world == 1 and args.e2e_graph:
        from kaolin_b200.render.mesh import make_graphed_dibr_rasterization
        a_fvz, a_fvi, a_ff, a_fnz = dev_in[0]
        fgraph = make_graphed_dibr_rasterization(H, W, a_fvz, a_fvi, a_ff, a_fnz, SIGMAINV, BOXLEN, KNUM)

        def step_graphed():
            with torch.no_grad():
                a_fvz.copy_(h_fvz, non_blocking=True); a_fvi.copy_(h_fvi, non_blocking=True)
                a_ff.copy_(h_ff, non_blocking=True); a_fnz.copy_(h_fnz, non_blocking=True)
            a_fvi.grad = None; a_ff.grad = None
            feat, soft, idx = fgraph(a_fvz, a_fvi, a_ff, a_fnz)
            torch.autograd.backward([feat, soft], [g_feat, g_soft])
            host_out[0][0].copy_(a_fvi.grad, non_blocking=True); host_out[0][1].copy_(a_ff.grad, non_blocking=True)
        for _ in range(3):
            step_graphed()
        torch.cuda.synchronize()
        start.record()
        for _ in range(args.steps):
            step_graphed()
        end.record(); torch.cuda.synchronize()
        gms = start.elapsed_time(end) / args.steps
        e2e_graphed = {"value": B * H * W / (gms * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": gms,
                       "api": "kaolin_b200.render.mesh.make_graphed_dibr_rasterization (forward and backward replayed "
                              "from CUDA graphs), same H2D / D2H as e2e, single-buffered"}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = peaks()
    A = algorithmic_bytes(B, F, H, W, D, s=2 if args.features == "bf16" else 4)
    ach = A["bwd_raster"] / (raster_bwd_ms * 1e-3) / 1e9
    traffic = None          # dram__bytes_read.sum + dram__bytes_write.sum of the same kernel (ncu --set full)
    traffic_src = None
    for prof_name in ("r2_kernels.json", "r1_kernels.json"):
        try:
            prof = json.load(open(os.path.join(ROOT, "profiles", prof_name)))
        except Exception:
            continue
        want = "raster_bwd_rows_kernel" if "raster_bwd_rows_kernel" in kernel_ms else "raster_bwd_kernel"
        for name, e in prof.items():
            if want in name and args.workload == "c4_shard" and args.features == "fp32":
                traffic = e.get("dram_traffic_bytes")
                traffic_src = f"profiles/{prof_name} (ncu --set full, c4_shard)"
        if traffic is not None:
            break
    # per-kernel table: CUDA-event time of every launch of one forward+backward (mean over the
    # traced steps) and, where the kernel has compulsory traffic of its own (SURVEY.md §8d split by
    # the kernel that moves it), algorithmic bytes -> GB/s -> fraction of the measured HBM peak
    sF = 2 if args.features == "bf16" else 4
    P_, NF_ = B * H * W, B * F
    alg = {
        "bin_faces_kernel<count>": NF_ * 28,                        # xy + validity
        "bin_faces_kernel<fill>": NF_ * (28 + 2 * 16),              # + one bin entry per set
        "dibr_tile_fwd_kernel": A["fwd"],                           # all per-pixel outputs + face reads
        "dibr_fwd2_kernel<S=2>": A["fwd"], "dibr_fwd2_kernel<S=1>": A["fwd"],
        "raster_bwd_rows_kernel": P_ * (D * sF + 8 + 12) + NF_ * (24 + 3 * D * sF),
        "raster_bwd_finalize_kernel": NF_ * (24 + 3 * D * 4),
        "raster_bwd_kernel": A["bwd_raster"],
        "soft_bwd_dense_kernel": band_px * 16 + NF_ * 24,           # soft, grad, idx of band pixels + grad_xy
        "soft_bwd_runs_kernel": band_px * 16 + NF_ * 24,
    }
    total_kernel_ms = sum(statistics.mean(v) for v in kernel_ms.values()) or 1.0
    kernels = []
    for name in kernel_order:
        ms = statistics.mean(kernel_ms[name])
        row = {"kernel": name, "ms": round(ms, 4), "share_of_kernel_time": round(ms / total_kernel_ms, 4)}
        if name in alg and ms > 0:
            gbs = alg[name] / (ms * 1e-3) / 1e9
            row.update({"algorithmic_bytes": int(alg[name]), "GBps": round(gbs, 1), "frac": round(gbs / peak, 4)})
        kernels.append(row)
    dominant = max(kernels, key=lambda r: r["ms"]) if kernels else None
    roofline = {
        "kernel": "rasterize backward scatter (the kernel BASELINE.json grades): dibr_b200_backward with only "
                  "grad_features = acc memset + raster_bwd_rows_kernel + raster_bwd_finalize_kernel "
                  "(warp-reduction raster_bwd_kernel + 2 output memsets when the row-walk path does not apply)",
        "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
        "traffic": traffic, "traffic_source": traffic_src,
        "peak_source": peak_src,
        "algorithmic_bytes_per_launch": A["bwd_raster"], "ms_per_launch": raster_bwd_ms,
        "kernels": kernels, "kernels_traced_steps": tsteps,
        "dominant_kernel": dominant,
        "phases": {
            "forward_ms": fwd_ms, "backward_ms": bwd_ms,
            "forward_GBps": A["fwd"] / (fwd_ms * 1e-3) / 1e9,
            "backward_GBps": A["bwd"] / (bwd_ms * 1e-3) / 1e9,
            "step_GBps": A["total"] / (ms_per_step * 1e-3) / 1e9,
            "step_frac_of_peak": A["total"] / (ms_per_step * 1e-3) / 1e9 / peak,
        },
    }
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "step_ms": step_stats, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": args.workload, "vertex_jitter": WORKLOADS[args.workload][5],
                   "views_per_gpu": B, "faces_per_view": F, "height": H,
                   "width": W, "feat_dim": D, "features": args.features, "cuda_graph": bool(args.graph and world == 1), "knum": KNUM, "sigmainv": SIGMAINV,
                   "boxlen": BOXLEN, "covered_fraction": covered,
                   "gather_transport": transport["used"] if world > 1 else None,
                   "parallelism": (f"views sharded x{world}; all-gather of per-view grads "
                                   + ({"peer": "by copy-engine stores into peer memory over NVLink (symmetric memory), ",
                                       "peer_sm": "by the dibr_b200_peer_push store kernel into peer memory over NVLink, ",
                                       "peer_mc": "by the dibr_b200_peer_push_multicast kernel (multimem.st through the "
                                                  "NVSwitch multicast mapping of the landing buffers), "}
                                      .get(transport["used"], "with NCCL, "))
                                   + (f"backward in {bwd_chunks} view chunks, chunk i's gathers overlap chunk i+1"
                                      if pipelined else
                                      "grad_face_features' gather overlapped with the soft-mask backward"
                                      if len(spans) == 1 else
                                      f"{len(spans)} view-chunks per step, chunk i's gather overlaps chunk i+1"))
                   if world > 1 else "single GPU",
                   "l2": "per-step working set (>1 GB of images) exceeds the 126 MB L2; no flush needed"},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": e2e_ms,
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "api": "kaolin_b200.render.mesh.dibr_rasterization + autograd, pinned host buffers; "
                       "uploads/downloads double-buffered on side streams",
                "d2h_contents": "the step's results as a training loop reads them: both gradients + the scalar "
                                "loss; the rendered images (features, soft_mask, face_idx: 28+ B/px) stay on the "
                                "device for the loss that consumes them - see e2e_images for the variant that "
                                "downloads them too",
                "host_wall_ms_per_step": wall_ms / args.steps},
        "e2e_images": e2e_images, "e2e_graphed": e2e_graphed,
        # kernels per (chunk of a) step, as traced, + the two push kernels of the peer-memory all-gather
        "gpu_launches": (max(1, len(kernel_order)) * len(spans)
                         + (2 if transport["used"] in ("peer_sm", "peer_mc") else 0)) * args.steps,
        "roofline": roofline,
        "triangle_pixel_tests_per_s": {
            "brute_force_equivalent": float(B) * H * W * F * 0.5 / (fwd_ms * 1e-3),
            "note": "faces x pixels the reference kernel would test (valid ~ F/2) / forward time"},
    }

    if not args.no_cpu_baseline and world == 1:
        s, cores, desc = cpu_sample(args.workload, args.cpu_seconds)
        t0 = time.perf_counter(); s.run(); dt = time.perf_counter() - t0
        line["cpu_baseline"] = {"value": s.pixels / dt / 1e6, "unit": UNIT, "cores": cores,
                                "kind": "port", "sample": desc, "seconds": dt,
                                "cores_detail": getattr(cpu_sample, "cores_info", None)}
    else:
        line["cpu_baseline"] = None

    if not args.no_ref_cuda and world == 1:
        line["reference_cuda"] = time_reference_cuda(args, dev, B, F, H, W, D, d_fvz, d_fvi, d_ff, d_fnz,
                                                     g_feat, g_soft)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


DUMP_BUDGET = 60 << 20     # bytes of all dumped arrays together (under 64 MB with the .npy headers)


def dump_outputs(out_dir, last_step):
    """Write what one resident step returned as <name>.npy: float32, face_idx as float64.  When the set
    exceeds DUMP_BUDGET, the images share one seeded sample of pixels and the gradients one of faces
    (rows of the flattened (B, H, W) / (B, F) leading dimensions, in increasing order), sized so that
    the set fits.  The same arguments give the same inputs and the same rows, so two builds can be
    compared output for output (the gradients accumulate with float atomics: compare them with a
    tolerance, the images bit for bit)."""
    import torch
    images, g_fvi, g_ff = last_step
    arrays = {"features": torch.cat([f for f, _, _ in images]), "soft_mask": torch.cat([s for _, s, _ in images]),
              "face_idx": torch.cat([i for _, _, i in images]),
              "grad_face_vertices_image": g_fvi, "grad_face_features": g_ff}
    lead = {n: 3 if n in ("features", "soft_mask", "face_idx") else 2 for n in arrays}
    rows = {n: t.shape[:lead[n]].numel() for n, t in arrays.items()}
    nbytes = sum(t.numel() * (8 if t.dtype == torch.int64 else 4) for t in arrays.values())
    keep = min(1.0, DUMP_BUDGET / max(nbytes, 1))
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        out = t.detach().reshape(rows[name], -1)
        if keep < 1.0:
            sel = np.random.default_rng(lead[name]).choice(rows[name], int(rows[name] * keep), replace=False)
            out = out[torch.from_numpy(np.sort(sel)).to(out.device)]
        out = out.to(torch.float64 if t.dtype == torch.int64 else torch.float32).cpu().numpy()   # bf16 too
        np.save(os.path.join(out_dir, name + ".npy"), out.reshape(t.shape) if keep >= 1.0 else out)


def time_reference_cuda(args, dev, B, F, H, W, D, d_fvz, d_fvi, d_ff, d_fnz, g_feat, g_soft):
    """The reference's own CUDA kernels (oracle/_ref, unmodified sources compiled for sm_100a)
    on a bounded number of views of the same workload, same GPU — the bar to beat."""
    import torch
    try:
        from oracle import ref_cuda
        if not ref_cuda.available():
            return {"unavailable": "oracle/_ref/kaolin_ref_C.so not present"}
        v = max(1, min(B, args.ref_cuda_views))
        a = (d_fvz[:v], d_fvi[:v], d_ff[:v].float(), d_fnz[:v], g_feat[:v].float().contiguous(),
             g_soft[:v].contiguous())
        ref_cuda.dibr_forward_backward(H, W, *a, SIGMAINV, BOXLEN, KNUM)
        torch.cuda.synchronize()
        n = 3
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(n):
            ref_cuda.dibr_forward_backward(H, W, *a, SIGMAINV, BOXLEN, KNUM)
        e.record()
        torch.cuda.synchronize()
        ms = s.elapsed_time(e) / n
        return {"value": v * H * W / (ms * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": ms,
                "sample": f"{v} of {B} views, reference wrappers restated in torch (oracle/ref_cuda.py)"}
    except Exception as exc:  # reported, never fatal for our arm
        return {"unavailable": f"{type(exc).__name__}: {exc}"}


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)

#!/usr/bin/env python
"""bench.py -- instance-field render throughput (BASELINE.json metric: Mrays/s; train-step ms @ 4096 rays) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload render|c4|train] [--rays R] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

Workload of the headline line (BASELINE.json configs[1], SURVEY.md section 8d "c2"): 640x480 frames (307 200 rays each) of the
synthetic 3D-FRONT-shaped room, bound 8 -> 4-cascade 128^3 occupancy grid, two 16-level 2^19-entry hash tables, 32 instance
classes, dt_gamma 1/128, max_steps 1024, T_thresh 1e-4; seeded random weights / tables (no network, no dataset).

A "step" = `world` frames rendered through NeRFNetwork.render (the call MaskTrainer.test_step makes, nerf/utils.py:1421): near/far
+ ONE fused launch (march + hash gathers x2 + tcgen05 MLP + composite) + the bg / depth tail.  Every step renders different
camera poses; L2 (126 MB) is flushed between timed steps by writing a 512 MB buffer (outside the per-step event pair).
At N > 1 rank r renders the interleaved row blocks r, r + N, ... of every frame of the step (cost follows marched samples, which
vary by +-25 % between poses) and the finished tiles are collected on rank 0 with ONE asynchronous NCCL gather per step that
overlaps the next step's render (the last step waits for its gather inside the timed region).

Keys of the JSON line:
  value        device-timed Mrays/s, rays resident in HBM (generated once by inerf_get_rays)
  e2e          the same through the public API from HOST inputs to HOST results: per step the camera poses (64 B each) go
               host->device, inerf_get_rays builds the rays on the device (as a reference user's get_rays does), the frame is
               rendered and every rank reads ITS OWN rows (image | depth | K logits) back to pinned host memory on a side
               stream (double buffered); ONE event pair brackets the whole region, L2 flushes and the last copy included
  roofline     the fused kernel's algorithmic gather bytes / its own CUDA-event time against the L2-RESIDENT read bandwidth
               measured in this run (instance_nerf_b200/probe.py): the 53 MB interleaved table lives in L2, HBM is not the
               binding roof (ncu: dram throughput 0.1 %).  `frac_of_hbm` keeps the round-1 figure, `gather_peak` the measured
               random 8-byte gather rate
  train_step   config c3 (4096 rays x max_steps 1024, one optimisation step as a CUDA graph), N = 1
  train_dp     config c5 (65 536 rays per GPU, data parallel, NCCL all-reduce of the gradient buffer inside the graph), every N
  cpu_baseline the reference's PyTorch (non-cuda_ray) renderer, restated in oracle/field_oracle.py and pinned against the
               reference's own outputs, on config c1 (160x120, K=16, 128 samples/ray: BASELINE.md B1), best of 3, host cores
  ref_cuda_path the reference's own CUDA kernels (oracle/_ref) on c2 and c3, timed in a subprocess (BASELINE.md B2)

--impl reference runs ONLY the CPU path (the reference arm): no CUDA code of this repo is touched.

--dump-outputs DIR (render workload) writes what NeRFNetwork.render returned in the last device-resident timed step -- on rank 0,
its own rows at N > 1 -- as DIR/<key>.npy (image, depth, instance_mask_logits; float32, 44 MB at K=32).  The inputs depend
only on the arguments, so two builds run with the same arguments can be compared output for output.
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
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "instance_field_render_Mrays_per_s"
UNIT = "Mrays/s"
W_IMG, H_IMG, K_INST, BOUND = 640, 480, 32, 8.0
DT_GAMMA, MAX_STEPS, T_THRESH = 1.0 / 128, 1024, 1e-4
N_POSES = 16
WORKLOAD = "c2: 640x480 instance-field render, 4x128^3 occupancy grid, 2x(16-level 2^19 hash grid), K=32, synthetic room"
WORKLOAD_C1 = "c1: 160x120 instance-field render, 128 uniform samples/ray, K=16, reference PyTorch (non-cuda_ray) path on CPU, synthetic room"
C1 = dict(H=120, W=160, K=16, T=128)
C4 = dict(H=1080, W=1920, frames=200)


def intrinsics(H=H_IMG, W=W_IMG):
    from instance_nerf_b200 import synthetic
    return synthetic.intrinsics(H, W)


def build_scene_and_model(device=None, K=K_INST, n_poses=N_POSES):
    import torch
    from instance_nerf_b200 import synthetic
    from instance_nerf_b200.nerf.network_mask import NeRFNetwork

    torch.manual_seed(0)
    model = NeRFNetwork(bound=BOUND, cuda_ray=True, num_instances=K, density_scale=1, density_thresh=10)
    synthetic.randomize_tables(model, 0)
    scene = synthetic.RoomScene(K, BOUND, 0)
    synthetic.install_scene(model, scene)
    poses = torch.from_numpy(synthetic.camera_poses(scene, n_poses, 1))
    if device is not None:
        model = model.to(device)
    return model.eval(), scene, poses


def train_batches(dev, scene, poses, n_rays, rank, world, n=8):
    """`n` training batches of `n_rays` rays as 8x8 patches (nerf/utils.py:83-100) with analytic first-hit labels; rays from the
    product's get_rays (one launch of inerf_get_rays per pose).  c3-sized batches (<= 8192 rays) come from ONE camera pose, as
    the reference's loader yields them (provider.py:635 batch_size 1); the large data-parallel batches (c5) take an equal share
    of patches from every pose, so that the marched-sample count -- which varies 2x between poses -- is the same mix on every
    rank and every step (weak scaling compares equal work per GPU)."""
    import numpy as np
    import torch
    from instance_nerf_b200.nerf.utils import get_rays

    out = []
    n_poses = poses.shape[0]
    for i in range(n):
        g = torch.Generator(device=dev).manual_seed(100 + i * world + rank)
        if n_rays <= 8192:
            sel, per = [(i * world + rank) % n_poses], n_rays
        else:
            sel, per = list(range(n_poses)), n_rays // n_poses
        os_, ds_ = [], []
        for p in sel:
            r = get_rays(poses[p][None].to(dev), intrinsics(), H_IMG, W_IMG, N=per, patch_size=8, generator=g)
            os_.append(r["rays_o"].reshape(-1, 3))
            ds_.append(r["rays_d"].reshape(-1, 3))
        o, d = torch.cat(os_).contiguous(), torch.cat(ds_).contiguous()
        labels = torch.from_numpy(scene.first_hit_labels(o.cpu().numpy().astype(np.float64), d.cpu().numpy().astype(np.float64)))
        out.append({"rays_o": o[None], "rays_d": d[None], "masks": labels[None].to(dev)})
    return out


# ------------------------------------------------------------------------------------------------ clocks --
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.idx)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        self.t.join(timeout=2)
        sm = sorted(float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit())
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 9 for n, v in zip(names, r[5:9]) if v.lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm)}


# ------------------------------------------------------------------------------------- CPU reference arm --
def make_cpu_reference(config: str = "c1", n_rays: int = 0):
    """The reference's PyTorch (non-cuda_ray) renderer -- NeRFMaskRenderer.run / staged render, mask_renderer.py:89-231,
    565-584 -- as restated in oracle/field_oracle.py (pinned against the reference's own outputs, tests/golden/ref_run.npz).
    config "c1": the whole 160x120 frame of the K=16 room (BASELINE.md B1); "c2-sample": `n_rays` rays strided over frame 0 of
    the c2 scene (K=32).  -> (render thunk, n_rays, samples_per_ray, cores)"""
    import torch
    from oracle import field_oracle as fo
    from oracle import host_oracle

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    if config == "c1":
        H, W, K, T = C1["H"], C1["W"], C1["K"], C1["T"]
    else:
        H, W, K, T = H_IMG, W_IMG, K_INST, 128
    model, _, poses = build_scene_and_model(None, K=K)
    sd = {k: v.detach().float().cpu() for k, v in model.state_dict().items()}
    field = fo.OracleField(sd, BOUND, K, density_scale=1.0)
    r = host_oracle.get_rays(poses[0:1], intrinsics(H, W), H, W)
    o, d = r["rays_o"].reshape(-1, 3).contiguous(), r["rays_d"].reshape(-1, 3).contiguous()
    if config != "c1":
        stride = max(1, o.shape[0] // n_rays)
        o, d = o[::stride][:n_rays].contiguous(), d[::stride][:n_rays].contiguous()

    def render():
        return field.render(o[None], d[None], max_ray_batch=4096, render_mask=True, num_steps=T, bg_color=1)

    return render, o.shape[0], T, cores


def time_cpu_reference(config, n_rays=0, warmup=1, repeats=3):
    render, n, T, cores = make_cpu_reference(config, n_rays)
    for _ in range(warmup):
        render()
    best = float("inf")
    for _ in range(repeats):
        t0 = time.perf_counter()
        render()
        best = min(best, time.perf_counter() - t0)
    return {"value": n / best / 1e6, "unit": UNIT, "cores": cores, "kind": "port", "rays": n, "samples_per_ray": T, "seconds_best": best,
            "repeats": repeats}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    render, n_rays, T, cores = make_cpu_reference("c1")
    for _ in range(max(1, args.warmup)):
        render()
    times = []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        render()
        times.append(time.perf_counter() - t0)
    total = sum(times)
    value = n_rays * args.steps / total / 1e6
    sample = (f"c1 = BASELINE.md B1: the whole 160x120 frame ({n_rays} rays) x {T} uniform samples/ray, K={C1['K']}, staged render in chunks of 4096 "
              f"rays, fp32, {cores} threads; mean of {args.steps} steps (best step {n_rays / min(times) / 1e6:.5f} Mrays/s)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": total / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": {"workload": WORKLOAD_C1, "rays_per_step": n_rays, "samples_per_ray": T,
                                        "note": "the reference's only CPU-runnable renderer is the non-cuda_ray path, whose config is c1 (BASELINE.json "
                                                "configs[0]); the GPU arm's headline config is c2"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if not args.no_c2_sample:
        c2 = time_cpu_reference("c2-sample", 8192, warmup=0, repeats=1)
        line["c2_scene_sample"] = {"value": c2["value"], "unit": UNIT, "sample": f"{c2['rays']} rays strided over frame 0 of the c2 scene (K=32), 128 uniform "
                                   f"samples/ray, {c2['seconds_best']:.1f} s", "cores": cores}
    emit(line)


# --------------------------------------------------------------------------------------------- GPU arm --
def _init_dist():
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        from datetime import timedelta
        dist.init_process_group("nccl", device_id=dev, timeout=timedelta(seconds=180))
    from instance_nerf_b200 import _lib
    _lib.lib()  # fail loudly if libinerf_b200.so is missing
    return rank, world, local_rank, dev


def run_gpu_arm(args):
    import torch
    import torch.distributed as dist
    from instance_nerf_b200 import parallel
    from instance_nerf_b200.nerf.utils import get_rays

    rank, world, local_rank, dev = _init_dist()
    model, scene, poses = build_scene_and_model(dev)
    N = H_IMG * W_IMG
    K = K_INST
    intr = intrinsics()
    # Work units of one step = `world` whole frames.  Rank r renders the row blocks r, r + world, ... of EVERY frame of the step
    # (H / world rows of each), not one frame of its own: cost is proportional to marched samples, which vary by +-25 % from
    # pose to pose, and the per-step tile gather is a synchronisation point -- interleaved rows give every rank the same mix
    # (SURVEY.md section 8e).  Rows stay whole, so the marcher's 32-ray patches remain runs of neighbouring pixels.
    block_rows = 4
    if H_IMG % (world * block_rows):
        raise SystemExit(f"bench.py: {H_IMG} rows do not split into {block_rows}-row blocks over {world} ranks")
    mine = parallel.shard_rows(H_IMG, W_IMG, rank, world, block_rows=block_rows).to(dev)    # this rank's pixel ids inside a frame
    n_groups = max(1, N_POSES // world)
    host_poses = [torch.stack([poses[(g * world + j) % N_POSES] for j in range(world)]).float().contiguous().pin_memory() for g in range(n_groups)]

    def rays_of(pose_group_dev):   # [world, 4, 4] on the device -> this rank's N rays of the step (ONE launch of inerf_get_rays)
        r = get_rays(pose_group_dev, intr, H_IMG, W_IMG, inds=mine if world > 1 else None)
        return r["rays_o"].view(-1, 3), r["rays_d"].view(-1, 3)

    dev_rays = [rays_of(p.to(dev)) for p in host_poses]
    kw = dict(staged=True, render_mask=True, perturb=False, dt_gamma=DT_GAMMA, max_steps=MAX_STEPS, T_thresh=T_THRESH, bg_color=1)
    flush_buf = torch.empty(512 * 1024 * 1024, dtype=torch.uint8, device=dev)
    # image 3 | depth 1 | logits K; double buffered so the NCCL gather of step i overlaps the render of step i + 1
    tiles = [torch.empty(N, 4 + K, dtype=torch.float32, device=dev) for _ in range(2)]
    gather = parallel.TileGather(N, 4 + K, dev, dst=0, depth=2)
    copy_done = [None, None]
    copy_stream = torch.cuda.Stream(device=dev)

    # kernel-only timing hook around the fused launch (events on the launching stream)
    kern_events, samples_seen = [], []
    launches = {"n": 0}
    fused = model._render_fused

    def timed_fused(*a, **k):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fused(*a, **k)
        e1.record()
        kern_events.append((e0, e1))
        samples_seen.append(model._work_counter.clone())
        launches["n"] += 3          # inerf_near_far_from_aabb + k_first_hit + k_render_fused
        return out

    model._render_fused = timed_fused

    def step(i, e2e=False, out_host=None):
        p = i % n_groups
        if e2e:
            o, d = rays_of(host_poses[p].to(dev, non_blocking=True))
            launches["n"] += 1      # k_get_rays
        else:
            o, d = dev_rays[p]
        b = gather.slot_ready() if not e2e else (i & 1)      # the gather that last used this buffer pair has finished (stream-side wait)
        if copy_done[b] is not None:      # ... and so has the device->host copy of the frame rendered two steps ago
            torch.cuda.current_stream().wait_event(copy_done[b])
            copy_done[b] = None
        tile = tiles[b]
        with torch.no_grad():
            r = model.render(o[None], d[None], **kw)
        tile[:, 0:3] = r["image"][0]
        tile[:, 3] = r["depth"][0]
        tile[:, 4:] = r["instance_mask_logits"][0]
        if e2e:
            # every rank reads ITS OWN rows back over its own PCIe link, on a side stream, so the copy of step i overlaps the
            # render of step i + 1 (double-buffered device tiles and pinned host buffers); no collective is needed for a result
            # that is wanted on the host
            ready = torch.cuda.Event()
            ready.record()
            copy_stream.wait_event(ready)
            with torch.cuda.stream(copy_stream):
                out_host[b].copy_(tile, non_blocking=True)
                copy_done[b] = torch.cuda.Event()
                copy_done[b].record()
        else:
            gather.submit(tile)
        return r

    def drain():
        gather.drain()
        for b in range(2):
            if copy_done[b] is not None:
                torch.cuda.current_stream().wait_event(copy_done[b])
                copy_done[b] = None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        step(i)
    drain()
    barrier()
    kern_events.clear(); samples_seen.clear(); launches["n"] = 0

    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()

    # ---- device-resident timed region: K steps, L2 flushed between them -----------------------------------------
    ev = []
    barrier()
    t_wall0 = time.perf_counter()
    torch.cuda.nvtx.range_push("inerf_timed")       # ncu --nvtx --nvtx-include "inerf_timed/" captures exactly these launches
    for i in range(args.steps):
        flush_buf.fill_(i & 0xFF)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        last = step(args.warmup + i)
        if i == args.steps - 1:
            drain()
        e1.record()
        ev.append((e0, e1))
    barrier()
    torch.cuda.nvtx.range_pop()
    wall_s = time.perf_counter() - t_wall0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)
    del last
    total_ms = sum(a.elapsed_time(b) for a, b in ev)
    kern_ms = [a.elapsed_time(b) for a, b in kern_events]
    n_samples = [int(s[2:4].view(torch.int64).item()) for s in samples_seen]
    n_tiles = [int(s[1].item()) for s in samples_seen]
    gpu_launches = launches["n"]

    # ---- end-to-end region: pinned host poses -> rays -> render -> pinned host results ----------------------------------
    out_host = [torch.empty(N, 4 + K, dtype=torch.float32).pin_memory() for _ in range(2)]
    for i in range(min(2, args.warmup)):
        step(i, True, out_host)
    drain()
    barrier()
    # one event pair around the whole region: L2 flushes and the final join of the copy stream are INSIDE it
    e2e0, e2e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2e0.record()
    for i in range(args.steps):
        flush_buf.fill_(i & 0xFF)
        step(args.warmup + i, True, out_host)
    drain()
    e2e1.record()
    barrier()
    e2e_ms = e2e0.elapsed_time(e2e1)
    clk = clocks.stop() if rank == 0 else None
    model._render_fused = fused

    if world > 1:
        t = torch.tensor([total_ms, e2e_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms, e2e_ms = float(t[0]), float(t[1])

    line = None
    if rank == 0:
        peaks = {}
        ppath = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(ppath):
            peaks = json.load(open(ppath))
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        # algorithmic bytes of the fused kernel (DESIGN.md "roofline"): per composited sample 2 tables x 16 levels x 8 corners x
        # 4 B (fp16 pair) = 1024 B of gathers; per ray 32 B in (o, d, near, far) + (5 + K) * 4 B out.  Nothing else touches HBM.
        avg_samples = sum(n_samples) / max(1, len(n_samples))
        alg_bytes = avg_samples * 1024.0 + N * (32.0 + (5 + K) * 4.0)
        avg_kern_ms = sum(kern_ms) / max(1, len(kern_ms))
        achieved = alg_bytes / (avg_kern_ms * 1e-3) / 1e9
        mlp_flops = avg_samples * (6144 + 12544 + 14208 + 128 * K)
        ms_per_step = total_ms / args.steps
        value = world * N / (ms_per_step * 1e-3) / 1e6
        try:
            from instance_nerf_b200 import probe
            l2 = probe.measure_l2_peaks(dev)
        except Exception as e:   # the probe library is a measurement helper: report its absence, do not lose the line
            l2 = {"error": f"{type(e).__name__}: {e}"}
        l2_peak = l2.get("l2_stream_gbs")
        prof = {}
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            try:
                prof = json.load(open(tpath))
            except Exception:
                prof = {}
        gathers_per_s = avg_samples * 128 / (avg_kern_ms * 1e-3)
        # What actually binds this kernel is the L1TEX tag stage: a warp's 32 8-byte gathers cost one lookup per distinct 32-byte
        # sector, and the probe's fully divergent gathers run at exactly 1 sector / clock / SM.  sectors / sample comes from the
        # committed ncu capture (l1tex__t_sectors_pipe_lsu_mem_global_op_ld.sum / composited samples), the peak from this run.
        spp = prof.get("k_render_fused_l1_sectors_per_sample")
        l1tex = None
        if spp and l2.get("gather_gps"):
            sect_s = avg_samples * spp / (avg_kern_ms * 1e-3)
            l1tex = {"sectors_per_sample": spp, "sectors_per_sample_source": prof.get("l1_sectors_source"), "achieved_gsectors_s": sect_s / 1e9,
                     "peak_gsectors_s": l2["gather_gps"] / 1e9, "frac": sect_s / l2["gather_gps"],
                     "what": "L1TEX sector (tag) lookups per second against the measured rate of fully divergent 8-byte gathers (1 sector / clock / SM)"}
        roof = {"kernel": "k_render_fused", "bound": "l2", "achieved": achieved, "unit": "GB/s", "traffic": prof.get("k_render_fused_dram_bytes_per_launch"),
                "peak": l2_peak if l2_peak else hbm_peak, "frac": achieved / (l2_peak if l2_peak else hbm_peak),
                "peak_source": ("measured in this run: coalesced 16-byte loads over an L2-resident 53 MB buffer (instance_nerf_b200/probe.py); the "
                                "interleaved fp16 table is L2-resident (ncu: lts hit rate 99.4 %, dram throughput 0.1 %).  8-byte gathers cannot "
                                "reach this figure: see l1tex (the binding unit) and gather_peak") if l2_peak else "L2 probe unavailable: HBM peak used",
                "kernel_ms": avg_kern_ms, "algorithmic_bytes_per_launch": alg_bytes, "gathers_per_s": gathers_per_s,
                "l1tex": l1tex,
                "gather_peak": {"gathers_per_s": l2.get("gather_gps"), "gbs_at_8B": l2.get("gather_gbs"),
                                "frac": gathers_per_s / l2["gather_gps"] if l2.get("gather_gps") else None,
                                "what": "random 8-byte ld.global.nc gathers from a 53 MB table at full occupancy (one sector per lane, no reuse): the "
                                        "access shape of the finest hashed levels; the coarse levels coalesce (several lanes per sector), so the "
                                        "kernel's gather rate exceeds it"},
                "frac_of_hbm": achieved / hbm_peak, "hbm_peak": hbm_peak,
                "hbm_peak_source": "MEASURED_PEAKS.json" if peaks else "fallback 6650 GB/s",
                "probe": l2, "mlp_tflops": mlp_flops / (avg_kern_ms * 1e-3) / 1e12}
        h2d = world * 64
        d2h = out_host[0].numel() * 4
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16 operands / f32 accumulate",
            "data": "synthetic",
            "config": {"workload": WORKLOAD, "rays_per_step_per_gpu": N, "samples_per_ray": avg_samples / N,
                       "tile_fill": (sum(n_samples) / max(1, 128 * sum(n_tiles))), "l2": "flushed between timed steps (512 MB write)",
                       "parallelism": (f"{world} frames per step, every frame's rows interleaved over {world} ranks (balanced by samples), async NCCL "
                                       f"gather of the finished row blocks to rank 0 overlapped with the next step "
                                       f"({N * (4 + K) * 4} B sent per rank per step over NVLink)") if world > 1 else "single GPU",
                       "wall_s_timed_region_incl_flush": wall_s},
            "e2e": {"value": world * N / (e2e_ms / args.steps * 1e-3) / 1e6, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "what": "poses (64 B each) host->device, rays built on the device by inerf_get_rays, render, own rows device->pinned host"},
            "gpu_launches": gpu_launches,
            "roofline": roof,
            "clocks": clk,
        }
    del flush_buf, tiles
    torch.cuda.empty_cache()

    # ---- training figures in the same run: c3 at N = 1, c5 (data parallel) at every N --------------------------------------
    if not args.no_train:
        if world == 1:
            try:
                tr = measure_train(dev, 0, 1, 20, 5, 4096, model, scene, poses)
            except Exception as e:   # the headline line must survive a failed graph capture: redo the figure eagerly and say so
                print(f"[bench] graphed train step failed ({type(e).__name__}: {e}); measuring the eager step", file=sys.stderr)
                torch.cuda.synchronize()
                os.environ["INERF_NO_GRAPH"] = "1"
                tr = measure_train(dev, 0, 1, 20, 5, 4096, model, scene, poses)
            if rank == 0:
                line["train_step"] = {"ms": tr["ms"], "ms_median": tr["ms_median"], "unit": "ms", "rays": 4096, "samples": tr["samples"],
                                      "workload": "c3: 4096 rays (8x8 patches) x max_steps 1024, K=32, fp16 autocast, CE + label smoothness, backward, Adam",
                                      "cuda_graph": tr["cuda_graph"], "graph_replays": tr["graph_replays"], "graph_captures": tr["graph_captures"]}
            try:   # stage-1 (RGB-sigma) training step, same rays: fused tcgen05 forward / backward vs the op-level kernels + cuBLAS autograd
                s1 = measure_train_rgb(dev, 20, 5, 4096, model, scene, poses)
                if rank == 0:
                    line["train_step_stage1"] = s1
            except Exception as e:
                print(f"[bench] stage-1 training figure failed ({type(e).__name__}: {e})", file=sys.stderr)
                if rank == 0:
                    line["train_step_stage1"] = {"error": f"{type(e).__name__}: {e}"}
        try:
            dp = measure_train(dev, rank, world, 12, 4, 65536, None, None, None)
            if rank == 0:
                line["train_dp"] = {"ms": dp["ms"], "ms_median": dp["ms_median"], "unit": "ms", "rays_per_gpu": 65536, "samples_per_gpu": dp["samples"],
                                    "rays_per_s": world * 65536 / (dp["ms"] * 1e-3), "n_gpus": world, "cuda_graph": dp["cuda_graph"],
                                    "graph_replays": dp["graph_replays"], "allreduce_bytes": dp["allreduce_bytes"], "allreduce_ms_alone": dp["allreduce_ms"],
                                    "workload": "c5: data-parallel instance-field training, 65536 rays/GPU (8x8 patches) x max_steps 1024, K=32, one NCCL "
                                                "all_reduce(SUM) of the flat gradient buffer inside the step, 1/N folded into the Adam pass"}
        except Exception as e:
            print(f"[bench] c5 data-parallel training figure failed ({type(e).__name__}: {e})", file=sys.stderr)
            if rank == 0:
                line["train_dp"] = {"error": f"{type(e).__name__}: {e}"}

    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            c1 = time_cpu_reference("c1", warmup=1, repeats=3)
            line["cpu_baseline"] = {"value": c1["value"], "unit": UNIT, "cores": c1["cores"], "kind": "port",
                                    "sample": f"c1 = BASELINE.md B1: whole 160x120 frame ({c1['rays']} rays) x 128 uniform samples/ray, K=16, reference "
                                              f"non-cuda_ray renderer (oracle port), 1 warm-up + best of 3: {c1['seconds_best']:.2f} s"}
        if world == 1 and not args.no_ref_cuda:
            line["ref_cuda_path"] = run_ref_cuda_subprocess()
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(out_dir, results):
    """results (a dict of [1, N, ...] device tensors, None for absent keys) -> out_dir/<key>.npy, float32."""
    import numpy as np
    arrays = {k: v[0].float().cpu().numpy() for k, v in results.items() if v is not None}
    total = sum(a.nbytes for a in arrays.values())
    if total > 64 << 20:
        raise SystemExit(f"bench.py: --dump-outputs would write {total} B, more than 64 MB")
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), a)


def run_ref_cuda_subprocess():
    """BASELINE.md B2: the reference's own CUDA kernels (oracle/_ref) on c2 / c3, in a separate process so that none of the
    checker's libraries are ever loaded next to the product's timed regions."""
    if not os.path.isdir(os.path.join(ROOT, "oracle", "_ref")) or not any(f.endswith(".so") for f in os.listdir(os.path.join(ROOT, "oracle", "_ref"))):
        return {"skipped": "oracle/_ref is not built (oracle/build_ref.sh needs /root/reference)"}
    try:
        r = subprocess.run([sys.executable, "-m", "oracle.ref_cuda_path", "--json", "--frames", "3", "--train-steps", "10"], cwd=ROOT,
                           capture_output=True, text=True, timeout=600)
        if r.returncode != 0:
            return {"skipped": f"oracle.ref_cuda_path exited {r.returncode}: {r.stderr[-300:]}"}
        return json.loads(r.stdout.strip().splitlines()[-1])
    except Exception as e:
        return {"skipped": f"{type(e).__name__}: {e}"}


# ---------------------------------------------------------------------------------------------- c4 arm --
def run_c4_arm(args):
    """BASELINE.json configs[3]: 1920x1080 multi-view render of 200 camera poses (the 3D-mask projection workload shape,
    scripts/project_3d_masks.py:135-266), whole frames round-robin over the ranks (parallel.shard_frames), one asynchronous NCCL
    gather of the finished frames to rank 0 per round.  A "step" = one round of `world` frames; rays are built on the device
    from the 64-byte pose of each frame."""
    import torch
    import torch.distributed as dist
    from instance_nerf_b200 import parallel, synthetic
    from instance_nerf_b200.nerf.utils import get_rays

    rank, world, local_rank, dev = _init_dist()
    H, W, n_frames = C4["H"], C4["W"], args.frames or C4["frames"]
    model, scene, _ = build_scene_and_model(dev)
    poses = torch.from_numpy(synthetic.camera_poses(scene, n_frames, 1)).to(dev)
    intr = intrinsics(H, W)
    N, K = H * W, K_INST
    kw = dict(staged=True, render_mask=True, perturb=False, dt_gamma=DT_GAMMA, max_steps=MAX_STEPS, T_thresh=T_THRESH, bg_color=1)
    # Frames differ in cost by +-25 %, and a gather is a rendezvous: with `depth` buffers a rank may run that many rounds ahead
    # of the slowest one before it has to wait (depth 2 measured 0.86 of linear at N = 8: every round waited for its slowest frame)
    depth = 2 if world == 1 else 6
    tiles = [torch.empty(N, 4 + K, dtype=torch.float32, device=dev) for _ in range(depth)]
    gather = parallel.TileGather(N, 4 + K, dev, dst=0, depth=depth)
    rounds = (n_frames + world - 1) // world
    # frame -> rank plan: equal frame counts, totals balanced by a cost estimate = samples marched by every 8th pixel of every 8th
    # row of each pose (one inerf_get_rays + one counting march per pose, ~0.2 ms; every rank computes the same plan, no
    # collective).  The estimate runs INSIDE the timed region.
    est_inds = ((torch.arange(0, H, 8, device=dev)[:, None] * W) + torch.arange(0, W, 8, device=dev)[None, :]).reshape(-1)

    def plan_frames():
        if world == 1:
            return list(range(n_frames))
        from instance_nerf_b200 import raymarching as rm
        counts = torch.zeros(n_frames, 2, dtype=torch.int32, device=dev)
        scratch = None
        for f in range(n_frames):
            r = get_rays(poses[f:f + 1], intr, H, W, inds=est_inds, aabb=model.aabb_infer, min_near=model.min_near)
            scratch = rm.count_samples(r["rays_o"], r["rays_d"], model.bound, model.density_bitfield, model.cascade, model.grid_size,
                                       r["nears"], r["fars"], counts[f], DT_GAMMA, MAX_STEPS, scratch)
        return parallel.balance_frames(counts[:, 0].tolist(), world)[rank]

    my_frames = plan_frames()

    def render_round(k):
        f = my_frames[k] if k < len(my_frames) else my_frames[-1]   # ranks past the end re-render their last frame (uniform collective)
        r = get_rays(poses[f:f + 1], intr, H, W)
        b = gather.slot_ready()
        with torch.no_grad():
            out = model.render(r["rays_o"], r["rays_d"], **kw)
        tile = tiles[b]
        tile[:, 0:3] = out["image"][0]
        tile[:, 3] = out["depth"][0]
        tile[:, 4:] = out["instance_mask_logits"][0]
        gather.submit(tile)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for k in range(min(3, rounds)):
        render_round(k)
    gather.drain()
    barrier()
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    my_frames = plan_frames()
    for k in range(rounds):
        render_round(k)
    gather.drain()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    samples = int(model._work_counter[2:4].view(torch.int64).item())
    clk = clocks.stop() if rank == 0 else None
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t[0])
    if rank == 0:
        value = n_frames * N / (ms * 1e-3) / 1e6
        emit({"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": rounds, "warmup": min(3, rounds), "ms_per_step": ms / rounds,
              "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f16 operands / f32 accumulate", "data": "synthetic",
              "config": {"workload": f"c4: {n_frames} camera poses x {W}x{H} instance-field render, K=32, whole frames over {world} GPU(s), equal counts, totals balanced by a marched-sample estimate",
                         "frames": n_frames, "rays_per_frame": N, "samples_per_ray_last_frame_rank0": samples / N,
                         "l2": "inputs larger than L2: every frame reads 2.07 M fresh rays and writes a 299 MB tile; tables stay L2-resident by design",
                         "parallelism": f"whole frames per rank (parallel.balance_frames), async NCCL gather of {N * (4 + K) * 4} B per frame to rank 0" if world > 1 else "single GPU"},
              "total_s": ms * 1e-3, "gpu_launches": 4 * rounds, "clocks": clk})
    if world > 1:
        dist.destroy_process_group()


def measure_train_rgb(dev, steps, warmup, n_rays, model, scene, poses):
    """Stage-1 (RGB-sigma) optimisation step, Trainer.train_step semantics (nerf/utils.py:536-632): a network with the instance
    model's sigma / colour tensors learns the colours that model renders for the same rays.  Timed twice: the fused path
    (inerf_field_forward_train_rgb / inerf_field_backward_rgb, whole step as a CUDA graph) and the reference's operator sequence on
    the op-level kernels + nn.Linear autograd (eager)."""
    import torch
    from instance_nerf_b200.nerf.network import NeRFNetwork
    from instance_nerf_b200.nerf.trainer import RGBTrainStep

    sd = {k: v for k, v in model.state_dict().items() if not (k.startswith("encoder_mask") or k.startswith("mask_net"))}
    kw = dict(dt_gamma=DT_GAMMA, max_steps=MAX_STEPS, T_thresh=T_THRESH)
    batches = train_batches(dev, scene, poses, n_rays, 0, 1, n=8)
    teacher = NeRFNetwork(bound=model.bound, cuda_ray=True, density_scale=model.density_scale, density_thresh=10)
    teacher.load_state_dict(sd)
    teacher = teacher.to(dev).eval()
    with torch.no_grad():
        for b in batches:
            b["images"] = teacher.render(b["rays_o"], b["rays_d"], staged=True, perturb=False, bg_color=1, **kw)["image"].clone()
            b.pop("masks")
    flush_buf = torch.empty(512 * 1024 * 1024, dtype=torch.uint8, device=dev)
    out = {"unit": "ms", "rays": n_rays,
           "workload": "stage-1 RGB-sigma step: 4096 rays x max_steps 1024, fp16 autocast, MSE, backward through compositing, both MLPs, SH "
                       "and the sigma hash table, Adam"}
    for tag, fused in (("fused", True), ("op_level", False)):
        student = NeRFNetwork(bound=model.bound, cuda_ray=True, density_scale=model.density_scale, density_thresh=10)
        student.load_state_dict(sd)
        student = student.to(dev)
        with torch.no_grad():
            student.encoder.embeddings.mul_(0.9)
        student.use_fused = fused
        tr = RGBTrainStep(student, lr=1e-3, fp16=True, patch_size=8, cuda_graph=fused and not os.environ.get("INERF_NO_GRAPH"), **kw)
        for i in range(max(warmup, 2 * len(batches))):
            tr.step(batches[i % 8])
        torch.cuda.synchronize()
        ev = []
        for i in range(steps):
            flush_buf.fill_(i & 0xFF)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            loss = tr.step(batches[(warmup + i) % 8])
            e1.record()
            ev.append((e0, e1))
        torch.cuda.synchronize()
        times = sorted(a.elapsed_time(b) for a, b in ev)
        out[tag] = {"ms": sum(times) / steps, "ms_median": times[len(times) // 2], "loss": float(loss.item()), "cuda_graph": bool(tr.cuda_graph),
                    "graph_replays": tr.graph_replays}
        del student, tr
    del flush_buf, teacher
    torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------- train arm --
def measure_train(dev, rank, world, steps, warmup, n_rays, model=None, scene=None, poses=None):
    """Times `steps` full optimisation steps (MaskTrainStep.step: render -> loss -> backward -> [all_reduce] -> Adam) with CUDA
    events, L2 flushed between steps.  -> dict(ms, samples, loss, clocks, ...)"""
    import torch
    import torch.distributed as dist
    from instance_nerf_b200.nerf.trainer import MaskTrainStep

    if model is None:
        model, scene, poses = build_scene_and_model(dev)
    use_graph = not os.environ.get("INERF_NO_GRAPH")
    trainer = MaskTrainStep(model, lr=1e-2, fp16=True, patch_size=8, label_regularization_weight=0.1, dt_gamma=DT_GAMMA, max_steps=MAX_STEPS,
                            T_thresh=T_THRESH, data_parallel=world > 1, cuda_graph=use_graph)
    batches = train_batches(dev, scene, poses, n_rays, rank, world, n=8)
    flush_buf = torch.empty(512 * 1024 * 1024, dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # every distinct batch goes through once before timing: the sample count differs per batch, and the first time a larger
    # sample stream shows up the caching allocator grows (cudaMalloc + sync) -- steady-state training never sees that
    for i in range(max(warmup, 2 * len(batches))):   # two passes: the second one replays a graph whose budget fits every batch
        trainer.step(batches[i % 8])
    barrier()
    model.step_counter.zero_()
    model.local_step = 0
    clocks = ClockSampler(dev.index or 0)
    if rank == 0:
        clocks.start()
    ev, totals = [], []
    torch.cuda.nvtx.range_push("inerf_timed")
    for i in range(steps):
        flush_buf.fill_(i & 0xFF)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        loss = trainer.step(batches[(warmup + i) % 8])
        e1.record()
        ev.append((e0, e1))
        totals.append(trainer.last_total)
    barrier()
    torch.cuda.nvtx.range_pop()
    times = sorted(a.elapsed_time(b) for a, b in ev)
    total_ms = sum(times)
    clk = clocks.stop() if rank == 0 else None
    n_samples = float(model.step_counter[: min(16, steps), 0].float().mean().item())
    if trainer.cuda_graph and trainer.graph_replays:
        n_samples = float(sum(totals)) / max(1, len(totals))
    ar_ms, ar_bytes = None, 0
    if world > 1:
        t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t[0])
        # the exchange on its own (same buffer, same collective), for the record: 10 back-to-back all-reduces
        ar_bytes = trainer.bucket.numel * 4
        barrier()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for _ in range(10):
            trainer.bucket.all_reduce()
        a1.record()
        barrier()
        ar_ms = a0.elapsed_time(a1) / 10
        trainer.bucket.flat.zero_()
    model.eval()
    for p in model.parameters():
        p.requires_grad_(True)
    del flush_buf
    return {"ms": total_ms / steps, "ms_median": times[len(times) // 2], "samples": n_samples, "loss": float(loss.item()), "clocks": clk,
            "cuda_graph": bool(trainer.cuda_graph), "graph_captures": trainer.graph_captures, "graph_replays": trainer.graph_replays,
            "allreduce_ms": ar_ms, "allreduce_bytes": ar_bytes}


def run_train_arm(args):
    """BASELINE.json configs[2] / [4]: instance-field training step (MaskTrainer.train_step + backward + Adam, nerf/utils.py:
    929-936, 1287-1373), `--rays` rays per GPU per step as 8x8 patches, max_steps 1024, fp16 autocast (the `-O` preset).
    At N > 1: data-parallel, one all_reduce of the flat mask-table + mask-net gradient buffer per step."""
    import torch.distributed as dist

    rank, world, local_rank, dev = _init_dist()
    n_rays = args.rays
    r = measure_train(dev, rank, world, args.steps, args.warmup, n_rays)
    if rank == 0:
        ms = r["ms"]
        cfg = "c3" if n_rays == 4096 and world == 1 else ("c5" if n_rays == 65536 else "train")
        line = {"metric": "instance_field_train_step_ms", "value": ms, "unit": "ms", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms, "higher_is_better": False, "scaling": "weak", "vs_baseline": None, "dtype": "f16 autocast / f32 params",
                "data": "synthetic",
                "config": {"workload": f"{cfg}: instance-field training step, {n_rays} rays/GPU (8x8 patches) x max_steps 1024, K=32, hash+MLP backward, Adam",
                           "rays_per_gpu": n_rays, "samples_per_step_per_gpu": r["samples"], "l2": "flushed between timed steps (512 MB write)",
                           "parallelism": f"dp{world}, one in-place all_reduce(SUM) of the flat gradient buffer, 1/N folded into Adam" if world > 1 else "single GPU",
                           "cuda_graph": r["cuda_graph"], "graph_replays": r["graph_replays"]},
                "ms_per_step_median": r["ms_median"], "rays_per_s": world * n_rays / (ms * 1e-3), "loss": r["loss"], "clocks": r["clocks"],
                "allreduce": {"bytes": r["allreduce_bytes"], "ms_alone": r["allreduce_ms"]}}
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def _claim_stdout():
    """The contract is ONE JSON line on stdout.  NCCL / CUDA libraries print banners ("NCCL version ...") straight to fd 1, so
    fd 1 is pointed at stderr for the life of the process and the JSON line goes out through a private duplicate."""
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


_JSON_OUT = None


def emit(line: dict):
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ref-cuda", action="store_true", help="skip the reference-CUDA-kernel figure (oracle/_ref subprocess) at N = 1")
    ap.add_argument("--no-c2-sample", action="store_true", help="reference arm: skip the extra c2-scene sample")
    ap.add_argument("--no-train", action="store_true", help="skip the train-step figures appended to the render line")
    ap.add_argument("--workload", default="render", choices=["render", "c4", "train"],
                    help="render = the headline metric on c2 (default); c4 = 200 poses x 1920x1080; train = train-step ms")
    ap.add_argument("--rays", type=int, default=4096, help="train workload: rays per GPU per step (4096 = config c3, 65536 = c5)")
    ap.add_argument("--frames", type=int, default=0, help="c4 workload: number of camera poses (default 200)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="render workload: write the render outputs of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 5 if args.impl == "reference" else 50
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload != "render"):
        ap.error("--dump-outputs applies to the render workload of --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        run_reference_arm(args)
    elif args.workload == "train":
        run_train_arm(args)
    elif args.workload == "c4":
        run_c4_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()

"""Volume extraction benchmark: NeRFRenderer.extract_volume (the fused inerf_extract_volume kernel) on the c2 synthetic scene
(bench.py's model: K = 32, bound 8, 4 x 128^3 occupancy grid), over its whole aabb_infer box at 256^3 and 512^3, dense
(skip_empty=False) and occupancy-gated, against the composed path a user has without it: inerf_volume_points -> forward_fused
([n, 32] fp32 logits to HBM) -> torch argmax / where (gated: the live voxels compacted with torch.nonzero first).  Every
call outputs sigma, rgb (one view direction) and label.

Prints ONE JSON line: card name and power limit, per (size, mode) the median ms over `--repeats` launches (one CUDA event pair
each, after warm-up), Mvoxels/s, the occupied fraction, and whether the two paths' outputs are identical (sigma and rgb bit for
bit, labels exactly).  L2 is NOT flushed between passes: the packed tables (2 x 16-level hash grid, fp16) are meant to stay
L2-resident, as within one bench.py step, and every pass writes 20 bytes per voxel of output, far more than L2 holds.

    python scripts/bench_extract.py [--sizes 256 512] [--repeats 20] [--no-composed]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

K = 32
VIEW_DIR = (0.0, 0.0, 1.0)
THRESH = 1.0


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = (s.strip() for s in out.split(",", 1))
        return name, power
    except Exception as e:   # the numbers still come out; the line says the card was not read
        return f"unknown ({e.__class__.__name__})", "unknown"


def timed(fn, repeats, warmup=3):
    import torch
    for _ in range(warmup):
        fn()
    ms = []
    for _ in range(repeats):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    ms.sort()
    return ms[len(ms) // 2], ms


def composed(m, n3, bbox, gated):
    """inerf_volume_points -> forward_fused -> torch rules: what extract_volume computes, with the [n, K] logits in HBM."""
    import numpy as np
    import torch
    from instance_nerf_b200._lib import call, ptr, stream_ptr
    X = Y = Z = n3
    n = X * Y * Z
    dev = m.aabb_infer.device
    xyzs = torch.empty(n, 3, dtype=torch.float32, device=dev)
    occ = torch.empty(n, dtype=torch.uint8, device=dev)
    bb = np.ascontiguousarray(bbox, dtype=np.float32)
    call("inerf_volume_points", bb.ctypes.data, X, Y, Z, ptr(m.density_bitfield) if gated else None, m.cascade, m.grid_size,
         float(m.bound), ptr(xyzs), ptr(occ), stream_ptr(dev))
    if gated:
        idx = occ.bool().nonzero().squeeze(1)
        xyzs = xyzs[idx]
    d = torch.tensor(VIEW_DIR, dtype=torch.float32, device=dev).expand(xyzs.shape[0], 3).contiguous()
    s, c, k = m.forward_fused(xyzs, d)
    s = s * float(m.density_scale)
    lab = torch.where(s >= THRESH, torch.argmax(k, dim=-1).to(torch.int32) + 1, 0)
    if not gated:
        return s.view(X, Y, Z), c.view(X, Y, Z, 3), lab.view(X, Y, Z)
    so = torch.zeros(n, dtype=torch.float32, device=dev)
    co = torch.zeros(n, 3, dtype=torch.float32, device=dev)
    lo = torch.zeros(n, dtype=torch.int32, device=dev)
    so[idx], co[idx], lo[idx] = s, c, lab
    return so.view(X, Y, Z), co.view(X, Y, Z, 3), lo.view(X, Y, Z)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[256, 512])
    ap.add_argument("--repeats", type=int, default=20)
    ap.add_argument("--no-composed", action="store_true", help="time the fused path only")
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_extract.py needs a CUDA device")
    sys.path.insert(0, ROOT)
    import bench
    from instance_nerf_b200 import _lib
    dev = torch.device("cuda:0")
    name, power = card()
    m, _, _ = bench.build_scene_and_model(dev, K=K)
    bbox = tuple(float(v) for v in m.aabb_infer.tolist())
    line = {"bench": "extract_volume", "card": name, "power_limit": power, "lib": os.path.basename(_lib.LIB_PATH), "K": K,
            "bbox": bbox, "outputs": "sigma, rgb, label", "sigma_thresh": THRESH, "repeats": args.repeats,
            "l2_flushed": False, "runs": []}
    with torch.no_grad():
        for n3 in args.sizes:
            nvox = n3 ** 3
            for gated in (False, True):
                call = lambda: m.extract_volume(n3, bbox=bbox, view_dir=VIEW_DIR, sigma_thresh=THRESH, skip_empty=gated)
                med, ms = timed(call, args.repeats)
                v = call()
                n_live = int(v["n_live"].item())
                run = {"size": n3, "mode": "gated" if gated else "dense", "voxels": nvox, "live_voxels": n_live,
                       "occupied_fraction": n_live / nvox if gated else None, "fused_ms": round(med, 4),
                       "fused_ms_min_max": [round(ms[0], 4), round(ms[-1], 4)], "fused_mvox_s": round(nvox / med / 1e3, 1)}
                if not args.no_composed:
                    cmed, _ = timed(lambda: composed(m, n3, bbox, gated), max(5, args.repeats // 2), warmup=1)
                    s, c, lab = composed(m, n3, bbox, gated)
                    run.update({"composed_ms": round(cmed, 4), "composed_mvox_s": round(nvox / cmed / 1e3, 1),
                                "speedup": round(cmed / med, 3),
                                "identical": bool(torch.equal(s.view(torch.int32), v["sigma"].view(torch.int32))
                                                  and torch.equal(c.view(torch.int32), v["rgb"].view(torch.int32))
                                                  and torch.equal(lab, v["label"]))})
                    del s, c, lab
                line["runs"].append(run)
                del v
                torch.cuda.empty_cache()
    print(json.dumps(line))


if __name__ == "__main__":
    main()

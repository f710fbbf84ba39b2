"""Mesh export benchmark: NeRFRenderer.extract_mesh's stages on the c2 synthetic scene (bench.py's model: K = 32, bound 8,
4 x 128^3 occupancy grid) over its whole aabb_infer box at 256^3 and 512^3, at threshold 10 (the reference's save_mesh default;
the synthetic field may have no density that high, and then the mesh is empty and only the count pass runs) and at the
median positive density of the volume, where there is a surface to emit.

Each stage is timed on its own with one CUDA event pair per run, median over `--repeats` runs after warm-up:
  extract_volume   sigma on the grid (fused kernel, occupancy-gated, no labels)
  count            inerf_mesh_count: per-sample masks and cases, tile totals, the two scans (occ::scan_block_counts)
  emit             inerf_mesh_emit: vertices and triangles
  attributes       the fused field forward at the vertices (rgb + logits), 1 + argmax, face labels
The marching-cubes passes are also stated as HBM traffic: the bytes they must move (the volume read once, the per-sample
state written and read back, the outputs written; reads of neighbouring samples are counted as cache hits, so this is a
lower bound) per sample, and that traffic over the pass time against the HBM copy bandwidth measured in the same run
(a 2 GiB device-to-device copy, read + write counted).  L2 is not flushed between runs; at 256^3 the 64 MiB volume fits
L2 (126 MB), at 512^3 (512 MiB) it does not.

Prints ONE JSON line with the card name and power limit.

    python scripts/bench_mesh.py [--sizes 256 512] [--repeats 20]
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

K = 32
THRESHOLD = 10.0
VIEW_DIR = (0.0, 0.0, 1.0)


def copy_peak_gbs(dev, repeats=10):
    """HBM bandwidth of a 2 GiB device-to-device copy (read + write), median of `repeats` timed copies."""
    import torch
    from bench_extract import timed
    n = 1 << 29
    a = torch.empty(n, dtype=torch.float32, device=dev).fill_(1.0)
    b = torch.empty_like(a)
    med, _ = timed(lambda: b.copy_(a), repeats)
    del a, b
    torch.cuda.empty_cache()
    return 2 * 4 * n / (med * 1e-3) / 1e9


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[256, 512])
    ap.add_argument("--repeats", type=int, default=20)
    args = ap.parse_args()
    if args.repeats < 20:
        raise SystemExit("--repeats must be at least 20")

    import numpy as np
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_mesh.py needs a CUDA device")
    import bench
    from bench_extract import card, timed
    from instance_nerf_b200._lib import call, lib, ptr, stream_ptr
    from instance_nerf_b200.mesh import face_labels
    dev = torch.device("cuda:0")
    name, power = card()
    m, _, _ = bench.build_scene_and_model(dev, K=K)
    bbox = tuple(float(v) for v in m.aabb_infer.tolist())
    bb = np.ascontiguousarray(bbox, dtype=np.float32)
    peak = copy_peak_gbs(dev)
    line = {"bench": "extract_mesh", "card": name, "power_limit": power, "K": K, "bbox": bbox,
            "repeats": args.repeats, "l2_flushed": False, "hbm_copy_peak_gbs": round(peak, 1), "runs": []}
    st = stream_ptr(dev)
    with torch.no_grad():
        for n3 in args.sizes:
            n = n3 ** 3
            vol = lambda: m.extract_volume(n3, bbox=bbox, sigma_thresh=0.0, skip_empty=True, labels=False)["sigma"]
            t_vol, _ = timed(vol, args.repeats)
            sigma = vol()
            scratch = torch.empty(int(lib().inerf_mesh_scratch_ints(n3, n3, n3)), dtype=torch.int32, device=dev)
            counts = torch.empty(2, dtype=torch.int32, device=dev)
            # the reference's default threshold, and one with a surface in any field: the median positive density
            for threshold in (THRESHOLD, float(sigma[sigma > 0].median()) / float(m.density_scale)):
                iso = threshold * float(m.density_scale)
                count = lambda: call("inerf_mesh_count", ptr(sigma), n3, n3, n3, iso, ptr(scratch), ptr(counts), st)
                t_count, _ = timed(count, args.repeats)
                V, F = counts.tolist()
                run = {"size": n3, "samples": n, "threshold": threshold, "iso": iso, "V": V, "F": F,
                       "extract_volume_ms": round(t_vol, 4), "count_ms": round(t_count, 4)}
                b_count = 4 * n + 4 * n                                   # v read, per-sample state written
                run.update({"count_bytes_per_sample": round(b_count / n, 2), "count_gbs": round(b_count / (t_count * 1e-3) / 1e9, 1),
                            "count_frac_of_copy_peak": round(b_count / (t_count * 1e-3) / 1e9 / peak, 3)})
                if F:
                    verts = torch.empty(V, 3, dtype=torch.float32, device=dev)
                    faces = torch.empty(F, 3, dtype=torch.int32, device=dev)
                    emit = lambda: call("inerf_mesh_emit", ptr(sigma), n3, n3, n3, bb.ctypes.data, iso, ptr(scratch), ptr(verts),
                                        ptr(faces), st)
                    t_emit, _ = timed(emit, args.repeats)
                    d = torch.empty_like(verts)
                    for a, c in enumerate(VIEW_DIR):
                        d[:, a] = c

                    def attrs():
                        _, rgb, logits = m.forward_fused(verts, d)
                        vl = torch.argmax(logits, dim=-1).to(torch.int32) + 1
                        return rgb, vl, face_labels(vl, faces)
                    t_attr, _ = timed(attrs, args.repeats)
                    # the same mesh as the public call, bit for bit
                    ref = m.extract_mesh(n3, bbox=bbox, threshold=threshold)
                    same = bool(torch.equal(ref["verts"].view(torch.int32), verts.view(torch.int32)) and torch.equal(ref["faces"], faces))
                    owners = int((scratch[:n] & 7 != 0).sum())
                    # state, v at the owners, vertices, first vertex of the owners (verts pass); state, faces (tris pass)
                    b_emit = 4 * n + 4 * owners + 12 * V + 4 * owners + 4 * n + 12 * F
                    run.update({"emit_ms": round(t_emit, 4), "attributes_ms": round(t_attr, 4),
                                "mc_share_of_total": round((t_count + t_emit) / (t_vol + t_count + t_emit + t_attr), 4),
                                "emit_bytes_per_sample": round(b_emit / n, 2), "emit_gbs": round(b_emit / (t_emit * 1e-3) / 1e9, 1),
                                "emit_frac_of_copy_peak": round(b_emit / (t_emit * 1e-3) / 1e9 / peak, 3),
                                "extract_mesh_identical": same})
                    del verts, faces, d, ref
                line["runs"].append(run)
            del sigma, scratch
            torch.cuda.empty_cache()
    print(json.dumps(line))


if __name__ == "__main__":
    main()

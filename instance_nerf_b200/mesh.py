"""Mesh export: marching cubes on the GPU (inerf_mesh_count / inerf_mesh_emit, csrc/mesh.cu) and a binary PLY writer.

mesh_from_volume   any CUDA float volume -> vertices and triangles (the geometry of extract_volume's voxel grid)
write_ply          binary little-endian PLY with optional per-vertex colour and instance label (numpy only)
save_mesh          the reference trainer's save_mesh(save_path, resolution, threshold) for a model, optionally one file per
                   instance

NeRFRenderer.extract_mesh composes extract_volume, mesh_from_volume and the field at the vertices."""
from __future__ import annotations

import os

import numpy as np
import torch

from ._lib import call, lib, ptr, stream_ptr


def mesh_from_volume(v: torch.Tensor, bbox, iso: float) -> dict:
    """The surface v = iso of a CUDA float32 volume v [X, Y, Z] (C order, every axis 2..2048) whose sample (i, j, k) sits at
    lo + (i, j, k) / (X, Y, Z) * (hi - lo), bbox = (lo xyz, hi xyz).  Inside is v > iso; normals point toward v < iso.

    -> {"verts": float32 [V, 3], "faces": int32 [F, 3]} on v's device, in a fixed order (include/inerf_b200.h).  Reads the
    two counts (8 bytes) once to size the outputs: the call's only host synchronisation."""
    if not (isinstance(v, torch.Tensor) and v.is_cuda and v.dtype == torch.float32 and v.dim() == 3):
        raise ValueError("mesh_from_volume takes a CUDA float32 volume [X, Y, Z]")
    v = v.contiguous()
    X, Y, Z = v.shape
    bb = np.ascontiguousarray(torch.as_tensor(bbox, dtype=torch.float32).reshape(6).tolist(), dtype=np.float32)
    dev = v.device
    n_scratch = int(lib().inerf_mesh_scratch_ints(X, Y, Z))
    scratch = torch.empty(max(n_scratch, 1), dtype=torch.int32, device=dev)
    counts = torch.empty(2, dtype=torch.int32, device=dev)
    st = stream_ptr(dev)
    call("inerf_mesh_count", ptr(v), X, Y, Z, float(iso), ptr(scratch), ptr(counts), st)
    n_verts, n_faces = counts.tolist()
    verts = torch.empty(n_verts, 3, dtype=torch.float32, device=dev)
    faces = torch.empty(n_faces, 3, dtype=torch.int32, device=dev)
    if n_faces:
        call("inerf_mesh_emit", ptr(v), X, Y, Z, bb.ctypes.data, float(iso), ptr(scratch), ptr(verts), ptr(faces), st)
    return {"verts": verts, "faces": faces}


def face_labels(vertex_label: torch.Tensor, faces: torch.Tensor) -> torch.Tensor:
    """Majority of a face's three vertex labels; the smallest when all three differ."""
    l = vertex_label[faces.long()]
    a, b, c = l[:, 0], l[:, 1], l[:, 2]
    return torch.where((a == b) | (a == c), a, torch.where(b == c, b, torch.minimum(a, torch.minimum(b, c))))


def _np(x):
    return x.detach().cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)


def rgb_to_u8(rgb) -> np.ndarray:
    """(x * 255) in fp32, clamped to [0, 255] and truncated, NaN -> 0: the quantisation of inerf_frame_to_u8."""
    s = np.asarray(rgb, np.float32) * np.float32(255.0)
    return np.nan_to_num(np.clip(s, 0.0, 255.0), nan=0.0).astype(np.uint8)


def write_ply(path, verts, faces, rgb=None, vertex_label=None) -> None:
    """Binary little-endian PLY: vertex x y z (float), red green blue (uchar, rgb in [0, 1]), label (int); face
    vertex_indices (uchar count 3, int)."""
    verts = _np(verts).astype(np.float32, copy=False).reshape(-1, 3)
    faces = _np(faces).astype(np.int32, copy=False).reshape(-1, 3)
    fields = [("x", "<f4"), ("y", "<f4"), ("z", "<f4")]
    props = ["property float x", "property float y", "property float z"]
    if rgb is not None:
        fields += [("red", "u1"), ("green", "u1"), ("blue", "u1")]
        props += ["property uchar red", "property uchar green", "property uchar blue"]
    if vertex_label is not None:
        fields += [("label", "<i4")]
        props += ["property int label"]
    vrec = np.empty(len(verts), dtype=fields)
    vrec["x"], vrec["y"], vrec["z"] = verts[:, 0], verts[:, 1], verts[:, 2]
    if rgb is not None:
        q = rgb_to_u8(_np(rgb).reshape(-1, 3))
        vrec["red"], vrec["green"], vrec["blue"] = q[:, 0], q[:, 1], q[:, 2]
    if vertex_label is not None:
        vrec["label"] = _np(vertex_label).reshape(-1)
    frec = np.empty(len(faces), dtype=[("n", "u1"), ("v", "<i4", (3,))])
    frec["n"] = 3
    frec["v"] = faces
    header = ["ply", "format binary_little_endian 1.0", f"element vertex {len(verts)}", *props, f"element face {len(faces)}",
              "property list uchar int vertex_indices", "end_header"]
    with open(path, "wb") as f:
        f.write(("\n".join(header) + "\n").encode("ascii"))
        f.write(vrec.tobytes())
        f.write(frec.tobytes())


def save_mesh(model, path, resolution=256, threshold=10, per_instance=False):
    """The reference's Trainer.save_mesh(save_path, resolution, threshold) for `model`: marching cubes over its density on a
    resolution^3 grid over aabb_infer, written as binary PLY.  An instance-field model also writes each vertex's label.
    per_instance: one file per face label instead, `<stem>_<label><ext>`, each with only its faces and their vertices
    (re-indexed), every vertex labelled with the file's label.  -> the paths written."""
    from .nerf.network import NeRFNetwork as RGBNetwork
    labels = per_instance or not isinstance(model, RGBNetwork)
    m = model.extract_mesh(resolution, threshold=threshold, labels=labels)
    verts, faces = m["verts"].cpu().numpy(), m["faces"].cpu().numpy()
    vl = m["vertex_label"].cpu().numpy() if labels else None
    if not per_instance:
        write_ply(path, verts, faces, vertex_label=vl)
        return [path]
    stem, ext = os.path.splitext(path)
    fl = m["face_label"].cpu().numpy()
    out = []
    for lab in np.unique(fl):
        sel = faces[fl == lab]
        used, inv = np.unique(sel.reshape(-1), return_inverse=True)
        p = f"{stem}_{int(lab)}{ext}"
        write_ply(p, verts[used], inv.reshape(-1, 3).astype(np.int32), vertex_label=np.full(len(used), lab, np.int32))
        out.append(p)
    return out

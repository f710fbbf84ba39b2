"""Mesh export on the GPU (instance_nerf_b200.mesh.mesh_from_volume -> inerf_mesh_count / inerf_mesh_emit, and
NeRFRenderer.extract_mesh): bit for bit against the C oracle (vertices and faces, same order) on analytic volumes and on a
density volume of the synthetic scene, run-to-run identity, the vertex attributes against the fused field forward, the
stage-1 network, the modular path, the single host read, and the PLY files of save_mesh."""
import warnings

import numpy as np
import pytest
import torch

from helpers import bits_equal
from ply_io import read_ply
from test_extract_gpu import SHAPE, SUB, VD, _points
from test_field_gpu import build_model

pytestmark = pytest.mark.gpu


def _analytic(name, shape=SHAPE):
    x, y, z = np.meshgrid(*[np.arange(n, dtype=np.float64) for n in shape], indexing="ij")
    c = [(n - 1) / 2 for n in shape]
    if name == "sphere":
        v = 81.0 - ((x - c[0]) ** 2 + (y - c[1]) ** 2 + (z - c[2]) ** 2)
    elif name == "torus":
        v = 16.0 - (np.sqrt((x - c[0]) ** 2 + (z - c[2]) ** 2) - 11.0) ** 2 - (y - c[1]) ** 2
    elif name == "two_spheres":
        v = np.maximum(49.0 - ((x - 9) ** 2 + (y - c[1]) ** 2 + (z - 12) ** 2), 36.0 - ((x - 27) ** 2 + (y - c[1]) ** 2 + (z - 38) ** 2))
    elif name == "noise":
        v = np.full(shape, -1.0)
        v[1:-1, 1:-1, 1:-1] = np.random.default_rng(3).standard_normal([n - 2 for n in shape])
    elif name == "linear":
        v = 0.3 * x - 0.7 * y + 0.45 * z
    elif name == "steps":            # values exactly at iso (0) and NaN samples
        v = np.floor(np.random.default_rng(4).random(shape) * 3) - 1
        v[np.random.default_rng(5).random(shape) < 0.02] = np.nan
    return v.astype(np.float32)


def _same(g, V, F):
    return bits_equal(g["verts"], V) and torch.equal(g["faces"].cpu(), torch.from_numpy(F))


@pytest.mark.parametrize("name,iso", [("sphere", 0.0), ("torus", 0.0), ("two_spheres", 0.0), ("noise", 0.0), ("noise", 0.7),
                                      ("linear", 1.3), ("steps", 0.0)])
def test_analytic_volumes_match_the_oracle(cuda, name, iso):
    from instance_nerf_b200.mesh import mesh_from_volume
    from oracle import mesh_oracle as mo
    v = _analytic(name)
    g = mesh_from_volume(torch.from_numpy(v).to(cuda), SUB, iso)
    V, F = mo.mesh(v, SUB, iso)
    assert len(F) > 0
    assert _same(g, V, F)


def _sigma_volume(m, shape=SHAPE, skip_empty=True):
    """extract_volume's sigma as extract_mesh takes it (occupancy-gated by default)"""
    return m.extract_volume(shape, bbox=SUB, sigma_thresh=0.0, skip_empty=skip_empty, labels=False)["sigma"]


def _median_sigma(m):
    """an iso level with surface around it: the median of the positive densities"""
    s = _sigma_volume(m)
    return float(s[s > 0].median())


def test_scene_density_matches_the_oracle_and_repeats(cuda):
    from instance_nerf_b200.mesh import mesh_from_volume
    from oracle import mesh_oracle as mo
    m, _ = build_model(cuda, 4)
    s = _sigma_volume(m)
    iso = _median_sigma(m)
    g1 = mesh_from_volume(s, SUB, iso)
    g2 = mesh_from_volume(s, SUB, iso)
    V, F = mo.mesh(s.cpu().numpy(), SUB, iso)
    assert len(F) > 1000
    assert _same(g1, V, F)
    assert bits_equal(g1["verts"], g2["verts"]) and torch.equal(g1["faces"], g2["faces"])


def test_vertex_with_t0_is_the_voxel_point(cuda):
    """In a 0 / 1 volume at iso 0, t is 0 (lower end outside at exactly iso) or 1 on every crossing edge, so every vertex is
    a voxel point of inerf_volume_points, bit for bit."""
    from instance_nerf_b200.mesh import mesh_from_volume
    m, _ = build_model(cuda, 2)
    v = (np.random.default_rng(6).random(SHAPE) < 0.3).astype(np.float32)
    g = mesh_from_volume(torch.from_numpy(v).to(cuda), SUB, 0.0)
    pts, _ = _points(m, SHAPE, SUB, bits=False)
    verts = g["verts"].cpu().numpy().view(np.uint32)
    pts = pts.cpu().numpy().view(np.uint32)
    assert len(verts) > 1000
    assert {tuple(p) for p in verts} <= {tuple(p) for p in pts}
    # a sample at 0 with a neighbour at 1 along an axis owns a vertex with t = 0 there: its own point
    X, Y, Z = SHAPE
    flat = v.reshape(-1)
    up = np.zeros(flat.shape, bool)
    for axis, step in enumerate((Y * Z, Z, 1)):
        idx = np.flatnonzero(np.indices(SHAPE)[axis].reshape(-1) + 1 < SHAPE[axis])
        up[idx] |= flat[idx + step] == 1
    owners = np.flatnonzero((flat == 0) & up)
    vset = {tuple(p) for p in verts}
    assert len(owners) > 100 and all(tuple(pts[e]) in vset for e in owners)


@pytest.mark.parametrize("K", [32, 2])
def test_vertex_attributes_equal_the_field(cuda, K):
    from instance_nerf_b200.mesh import face_labels
    m, _ = build_model(cuda, K)
    thr = _median_sigma(m)
    r = m.extract_mesh(SHAPE, bbox=SUB, threshold=thr, view_dir=VD)
    V = r["verts"]
    assert V.shape[0] > 1000 and r["iso"] == thr
    s, c, k = m.forward_fused(V, torch.tensor(VD, device=cuda).expand(V.shape[0], 3).contiguous())
    assert bits_equal(r["rgb"], c)
    assert torch.equal(r["vertex_label"], torch.argmax(k, dim=-1).to(torch.int32) + 1)
    # face label: majority of the three vertex labels, the smallest when all differ
    l = r["vertex_label"].cpu().numpy()[r["faces"].cpu().numpy()]
    exp = np.array([min(t) if len(set(t)) == 3 else max(set(t), key=list(t).count) for t in l.tolist()], np.int32)
    assert np.array_equal(r["face_label"].cpu().numpy(), exp)
    assert torch.equal(face_labels(r["vertex_label"], r["faces"]), r["face_label"])
    assert len(np.unique(l)) > 1
    # the mesh is the one of the density volume at iso = threshold * density_scale
    from instance_nerf_b200.mesh import mesh_from_volume
    g = mesh_from_volume(_sigma_volume(m), SUB, thr)
    assert bits_equal(g["verts"], V) and torch.equal(g["faces"], r["faces"])
    assert "rgb" not in m.extract_mesh(SHAPE, bbox=SUB, threshold=thr)


def test_threshold_is_scaled_by_density_scale(cuda):
    m, _ = build_model(cuda, 4, density_scale=25.0)
    thr = _median_sigma(m) / 25.0
    r = m.extract_mesh(SHAPE, bbox=SUB, threshold=thr, labels=False)
    assert r["iso"] == thr * 25.0 and r["faces"].shape[0] > 1000 and "vertex_label" not in r


def test_stage1_network(cuda):
    from helpers import scene_arrays
    from instance_nerf_b200 import synthetic
    from instance_nerf_b200.nerf.network import NeRFNetwork
    from oracle import mesh_oracle as mo
    torch.manual_seed(0)
    m = NeRFNetwork(bound=8.0, cuda_ray=True, density_scale=3.0, density_thresh=10)
    synthetic.randomize_tables(m, 0)
    _, _, grid, bits = scene_arrays(16, 8.0, 0)
    with torch.no_grad():
        m.density_grid.copy_(torch.from_numpy(grid)); m.density_bitfield.copy_(torch.from_numpy(bits))
    m = m.to(cuda).eval()
    with pytest.raises(ValueError):
        m.extract_mesh(16)
    s = _sigma_volume(m, skip_empty=False)
    thr = float(s.median()) / 3.0
    r = m.extract_mesh(SHAPE, bbox=SUB, threshold=thr, view_dir=VD, labels=False, skip_empty=False)
    assert "vertex_label" not in r and "face_label" not in r
    V, F = mo.mesh(s.cpu().numpy(), SUB, thr * 3.0)
    assert len(F) > 1000 and _same(r, V, F)
    with torch.no_grad():
        _, c = m(r["verts"], torch.tensor(VD, device=cuda).expand(len(V), 3).contiguous())
    assert bits_equal(r["rgb"], c)


def test_modular_path(cuda):
    """use_fused = False: extract_volume's modular path gives sigma, the network's forward under fp16 autocast gives the
    vertex fields; the mesh is the oracle's mesh of that sigma volume, the labels agree with the fused field."""
    from oracle import mesh_oracle as mo
    m, _ = build_model(cuda, 16)
    thr = _median_sigma(m)
    m.use_fused = False
    try:
        s = _sigma_volume(m)
        r = m.extract_mesh(SHAPE, bbox=SUB, threshold=thr, view_dir=VD)
    finally:
        m.use_fused = True
    V, F = mo.mesh(s.cpu().numpy(), SUB, thr)
    assert len(F) > 1000 and _same(r, V, F)
    _, c, k = m.forward_fused(r["verts"], torch.tensor(VD, device=cuda).expand(len(V), 3).contiguous())
    agree = float((r["vertex_label"] == torch.argmax(k, dim=-1).to(torch.int32) + 1).float().mean())
    assert agree >= 0.99, agree
    torch.testing.assert_close(r["rgb"], c, rtol=0, atol=2e-3)


def test_extract_mesh_reads_the_device_once(cuda):
    m, _ = build_model(cuda, 32)
    m.extract_mesh(SHAPE, bbox=SUB, threshold=1.0, view_dir=VD)      # packs tables / weights, loads the module
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("warn")
    try:
        with warnings.catch_warnings(record=True) as w:
            warnings.simplefilter("always")
            r = m.extract_mesh(SHAPE, bbox=SUB, threshold=1.0, view_dir=VD)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    syncs = [x for x in w if "synchroniz" in str(x.message).lower()]
    assert len(syncs) == 1, [str(x.message) for x in w]
    assert r["faces"].shape[0] > 0


def test_ply_files(cuda, tmp_path):
    from instance_nerf_b200.mesh import rgb_to_u8, save_mesh, write_ply
    m, _ = build_model(cuda, 8)
    r = m.extract_mesh(SHAPE, bbox=SUB, threshold=_median_sigma(m), view_dir=VD)
    p = tmp_path / "scene.ply"
    write_ply(p, r["verts"], r["faces"], rgb=r["rgb"], vertex_label=r["vertex_label"])
    back = read_ply(p)
    assert np.array_equal(back["verts"].view(np.uint32), r["verts"].cpu().numpy().view(np.uint32))
    assert np.array_equal(back["faces"], r["faces"].cpu().numpy())
    assert np.array_equal(back["rgb"], rgb_to_u8(r["rgb"].cpu().numpy()))
    assert np.array_equal(back["label"], r["vertex_label"].cpu().numpy())

    # save_mesh: the reference's entry point over aabb_infer; per instance, one file per face label
    thr = 1.0
    whole = save_mesh(m, str(tmp_path / "all.ply"), resolution=40, threshold=thr)
    full = read_ply(whole[0])
    ref = m.extract_mesh(40, threshold=thr)
    assert np.array_equal(full["faces"], ref["faces"].cpu().numpy()) and np.array_equal(full["label"], ref["vertex_label"].cpu().numpy())
    parts = save_mesh(m, str(tmp_path / "obj.ply"), resolution=40, threshold=thr, per_instance=True)
    fl = ref["face_label"].cpu().numpy()
    assert len(parts) == len(np.unique(fl)) > 1

    def tri_keys(verts, faces):
        t = verts[faces].reshape(len(faces), 9).view(np.uint32)
        return sorted(map(tuple, t.tolist()))
    union = []
    for path in parts:
        d = read_ply(path)
        labs = np.unique(d["label"])
        assert len(labs) == 1 and path.endswith(f"_{int(labs[0])}.ply")
        assert len(np.unique(d["faces"])) == len(d["verts"])            # re-indexed: every vertex is used
        assert len(d["faces"]) == int((fl == labs[0]).sum())
        union += tri_keys(d["verts"], d["faces"])
    assert sorted(union) == tri_keys(full["verts"], full["faces"])

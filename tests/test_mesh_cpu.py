"""CPU suite for the mesh export: the generated marching-cubes table (against its rule, case by case), the C oracle on
analytic volumes (closed, oriented surfaces with the right topology and volume), and argument validation of
inerf_mesh_count / inerf_mesh_emit, which returns its negative inerf_status before any launch."""
import importlib.util
import os
import re
from collections import Counter

import numpy as np
import pytest

from instance_nerf_b200 import _lib
from oracle import mesh_oracle as mo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "instance_nerf_b200", "csrc", "mc_table.h")


def _gen():
    spec = importlib.util.spec_from_file_location("gen_mc_table", os.path.join(ROOT, "scripts", "gen_mc_table.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def _header_table():
    """(edge corners [12, 2], triangle count [256], triangle edges per case) parsed from the checked-in header."""
    text = open(HEADER).read()

    def body(name):
        return [int(x) for x in re.findall(r"-?\d+", text.split(name, 1)[1].split("=", 1)[1].split("};", 1)[0])]

    edges = np.array(body("MC_EDGE_CORNERS[12][2]"), int).reshape(12, 2)
    count = np.array(body("MC_TRI_COUNT[256]"), int)
    rows = np.array(body("MC_TRI_TABLE[256][16]"), int).reshape(256, 16)
    tris = [[tuple(rows[c, 3 * t:3 * t + 3]) for t in range(count[c])] for c in range(256)]
    for c in range(256):
        assert (rows[c, 3 * count[c]:] == -1).all()
    return edges, count, tris


def test_generator_output_equals_header():
    assert _gen().render(_gen().table()) == open(HEADER).read()


def test_edges():
    edges, _, _ = _header_table()
    for e, (a, b) in enumerate(edges):
        assert a < b and a ^ b == 1 << (e // 4)   # lower corner first, along axis e // 4
    assert len({tuple(x) for x in edges}) == 12


def _face_rule_segments(case, edges):
    """Undirected segments of the face rule, restated: on each face, each cyclic run of inside corners is cut off by a
    segment between the two crossing edges bounding it."""
    eid = {frozenset(map(int, ab)): i for i, ab in enumerate(edges)}
    segs = Counter()
    for axis in range(3):
        u, w = [b for b in range(3) if b != axis]
        for s in (0, 1):
            ring = [(s << axis) | (cu << u) | (cw << w) for cu, cw in ((0, 0), (1, 0), (1, 1), (0, 1))]
            ins = [bool(case >> c & 1) for c in ring]
            crossing = [eid[frozenset((ring[i], ring[(i + 1) % 4]))] for i in range(4) if ins[i] != ins[(i + 1) % 4]]
            if len(crossing) == 2:
                segs[frozenset(crossing)] += 1
            elif len(crossing) == 4:   # ambiguous face: each inside corner alone
                for i in range(4):
                    if ins[i]:
                        segs[frozenset((eid[frozenset((ring[i - 1], ring[i]))], eid[frozenset((ring[i], ring[(i + 1) % 4]))]))] += 1
    return segs


def test_every_case_follows_the_rule():
    edges, count, tris = _header_table()
    assert count[0] == 0 and count[255] == 0 and count.max() <= 5
    assert np.bincount(count, minlength=6).tolist() == [2, 16, 50, 80, 76, 32]
    for case in range(256):
        inside = [bool(case >> c & 1) for c in range(8)]
        crossing = {e for e, (a, b) in enumerate(edges) if inside[a] != inside[b]}
        used = {e for t in tris[case] for e in t}
        assert used == crossing, case
        uses = Counter(frozenset(p) for t in tris[case] for p in ((t[0], t[1]), (t[1], t[2]), (t[2], t[0])))
        boundary = Counter({k: 1 for k, n in uses.items() if n % 2})
        assert boundary == _face_rule_segments(case, edges), case
        assert all(len(set(t)) == 3 for t in tris[case]), case


# ---- the oracle on analytic volumes ----------------------------------------------------------------------------------------

def _edges(F):
    return np.concatenate([F[:, [0, 1]], F[:, [1, 2]], F[:, [2, 0]]])


def _directed_matched(F):
    d = Counter(map(tuple, _edges(F)))
    return all(d.get((b, a), 0) == n for (a, b), n in d.items())


def _euler(V, F):
    und = {tuple(sorted(e)) for e in _edges(F)}
    return len(np.unique(F)) - len(und) + len(F)


def _signed_volume(V, F):
    a, b, c = (V[F[:, i]].astype(np.float64) for i in range(3))
    return float(np.einsum("ij,ij->i", a, np.cross(b, c)).sum() / 6)


def _components(F):
    parent = list(range(int(F.max()) + 1))

    def find(x):
        while parent[x] != x:
            parent[x] = parent[parent[x]]
            x = parent[x]
        return x
    for a, b, c in F:
        for p, q in ((a, b), (b, c)):
            parent[find(p)] = find(q)
    return len({find(x) for x in np.unique(F)})


def _grid(shape):
    return np.meshgrid(*[np.arange(n, dtype=np.float64) for n in shape], indexing="ij")


def test_sphere():
    R, r = 40, 12.3
    x, y, z = _grid((R, R, R))
    v = (r * r - ((x - 19.5) ** 2 + (y - 19.2) ** 2 + (z - 19.7) ** 2)).astype(np.float32)
    V, F = mo.mesh(v, (0, 0, 0, R, R, R), 0.0)
    und = Counter(tuple(sorted(e)) for e in _edges(F))
    assert set(und.values()) == {2}                       # every index edge used exactly twice
    assert set(Counter(map(tuple, _edges(F))).values()) == {1} and _directed_matched(F)
    assert _euler(V, F) == 2 and _components(F) == 1
    vol = _signed_volume(V, F)
    assert vol > 0 and abs(vol / (4 / 3 * np.pi * r ** 3) - 1) < 0.01
    assert len(np.unique(F)) == len(V)                    # every vertex is used


def test_torus():
    x, y, z = _grid((48, 48, 32))
    R0, r0 = 12.0, 5.0
    q = np.sqrt((x - 23.5) ** 2 + (y - 23.5) ** 2) - R0
    v = (r0 * r0 - q ** 2 - (z - 15.5) ** 2).astype(np.float32)
    V, F = mo.mesh(v, (-1, -1, -1, 1, 1, 1), 0.0)
    assert _euler(V, F) == 0 and _directed_matched(F) and _signed_volume(V, F) > 0


def test_two_spheres():
    x, y, z = _grid((40, 24, 24))
    a = 36.0 - ((x - 10) ** 2 + (y - 12) ** 2 + (z - 12) ** 2)
    b = 25.0 - ((x - 28) ** 2 + (y - 11) ** 2 + (z - 12.5) ** 2)
    v = np.maximum(a, b).astype(np.float32)
    V, F = mo.mesh(v, (0, 0, 0, 4, 2.4, 2.4), 0.0)
    assert _components(F) == 2 and _euler(V, F) == 4 and _directed_matched(F)


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_padded_noise_is_a_closed_two_cycle(seed):
    rng = np.random.default_rng(seed)
    v = np.full((24, 24, 24), -1.0, np.float32)
    v[1:-1, 1:-1, 1:-1] = rng.standard_normal((22, 22, 22)).astype(np.float32)
    V, F = mo.mesh(v, (0, 0, 0, 1, 1, 1), 0.0)
    assert len(F) > 1000 and _directed_matched(F)
    assert np.isfinite(V).all()


def test_linear_field_lies_on_the_plane():
    shape = (20, 17, 23)
    bb = np.array([-0.5, 0.25, -1.0, 0.75, 1.5, 0.5], np.float32)
    pts = [bb[a] + np.arange(n, dtype=np.float64) / n * (bb[3 + a] - bb[a]) for a, n in enumerate(shape)]
    x, y, z = np.meshgrid(*pts, indexing="ij")
    n = np.array([0.3, -0.7, 0.5])
    iso = -0.41
    V, F = mo.mesh((n[0] * x + n[1] * y + n[2] * z).astype(np.float32), bb, iso)
    assert len(F) > 100
    np.testing.assert_allclose(V.astype(np.float64) @ n, iso, rtol=0, atol=1e-5)
    # normals point toward low values: against the gradient n
    a, b, c = (V[F[:, i]].astype(np.float64) for i in range(3))
    assert (np.cross(b - a, c - a) @ n < 0).all()


def test_uniform_volumes_are_empty():
    for val in (1.0, -1.0, np.nan):
        V, F = mo.mesh(np.full((5, 6, 7), val, np.float32), (0, 0, 0, 1, 1, 1), 0.0)
        assert V.shape == (0, 3) and F.shape == (0, 3)


def test_values_equal_to_iso_count_as_outside():
    v = np.zeros((6, 6, 6), np.float32)
    v[2:4, 2:4, 2:4] = 0.5
    V, F = mo.mesh(v, (0, 0, 0, 1, 1, 1), 0.5)            # the block equals iso: nothing is inside
    assert len(F) == 0
    V, F = mo.mesh(v, (0, 0, 0, 1, 1, 1), 0.0)            # zeros equal iso: outside; the block is inside
    assert len(F) > 0 and np.isfinite(V).all() and _directed_matched(F)
    # every vertex sits on an outside sample (t = 1 from the block: iso - 0.5 over 0 - 0.5 -> 1), i.e. on the lattice
    assert np.array_equal(V * 6, np.round(V * 6))


def test_nan_samples_give_defined_vertices():
    v = np.zeros((5, 5, 5), np.float32)
    v[2, 2, 2] = np.nan
    v[1:4, 1:4, 3] = 1.0
    V, F = mo.mesh(v, (0, 0, 0, 1, 1, 1), 0.5)
    assert len(F) > 0 and np.isfinite(V).all() and _directed_matched(F)


# ---- argument validation of the C ABI --------------------------------------------------------------------------------------

NULL_, SIZE = -1, -2
FAKE = 0x10000   # a non-NULL "device" pointer: every call below is rejected before anything dereferences it
GOOD = np.array([-1, -1, -1, 1, 1, 1], np.float32)


@pytest.fixture(scope="module")
def L():
    if not os.path.exists(_lib.LIB_PATH):
        _lib.build()
    return _lib.lib()


def _count(L, X=8, Y=8, Z=8, v=FAKE, scratch=FAKE, counts=FAKE):
    return L.inerf_mesh_count(v, X, Y, Z, 0.5, scratch, counts, None)


def _emit(L, X=8, Y=8, Z=8, v=FAKE, bbox=GOOD, scratch=FAKE, verts=FAKE, tris=FAKE):
    return L.inerf_mesh_emit(v, X, Y, Z, None if bbox is None else bbox.ctypes.data, 0.5, scratch, verts, tris, None)


@pytest.mark.parametrize("X,Y,Z", [(1, 8, 8), (8, 1, 8), (8, 8, 1), (0, 8, 8), (2049, 8, 8), (8, 8, 2049),
                                   (2048, 2048, 512),      # X * Y * Z = 2^31
                                   (1024, 1024, 683),      # 3 X Y Z >= 2^31: more vertices than int32 could index
                                   (800, 800, 800)])       # 5 (X-1)(Y-1)(Z-1) >= 2^31: more triangles than int32 counts
def test_bad_sizes(L, X, Y, Z):
    assert _count(L, X, Y, Z) == SIZE
    assert _emit(L, X, Y, Z) == SIZE
    assert L.inerf_mesh_scratch_ints(X, Y, Z) == 0


@pytest.mark.parametrize("bbox", [
    np.array([-1, -1, -1, -1, 1, 1], np.float32),     # hi == lo
    np.array([-1, 2, -1, 1, 1, 1], np.float32),       # hi < lo
    np.array([-1, -1, -1, 1, np.nan, 1], np.float32),
    np.array([-np.inf, -1, -1, 1, 1, 1], np.float32),
    np.array([-1, -1, -1, 1, 1, np.inf], np.float32),
])
def test_bad_bbox(L, bbox):
    assert _emit(L, bbox=bbox) == SIZE


def test_null_pointers(L):
    assert _count(L, v=None) == NULL_
    assert _count(L, scratch=None) == NULL_
    assert _count(L, counts=None) == NULL_
    for kw in ("v", "bbox", "scratch", "verts", "tris"):
        assert _emit(L, **{kw: None}) == NULL_, kw


@pytest.mark.parametrize("X,Y,Z", [(2, 2, 2), (37, 20, 53), (256, 256, 256), (512, 512, 512), (2048, 2048, 100)])
def test_scratch_formula(L, X, Y, Z):
    # per-sample state and first vertex | vertex and triangle counts per 1024-sample tile
    n = X * Y * Z
    assert L.inerf_mesh_scratch_ints(X, Y, Z) == 2 * n + 2 * ((n + 1023) // 1024)


def test_write_ply_round_trip(tmp_path):
    from instance_nerf_b200.mesh import rgb_to_u8, write_ply
    from ply_io import read_ply
    rng = np.random.default_rng(0)
    V = rng.standard_normal((50, 3)).astype(np.float32)
    F = rng.integers(0, 50, (70, 3)).astype(np.int32)
    rgb = rng.random((50, 3)).astype(np.float32)
    rgb[0] = [np.nan, -0.5, 1.5]
    lab = rng.integers(0, 9, 50).astype(np.int32)
    p = tmp_path / "m.ply"
    write_ply(p, V, F, rgb=rgb, vertex_label=lab)
    r = read_ply(p)
    assert np.array_equal(r["verts"], V) and np.array_equal(r["faces"], F) and np.array_equal(r["label"], lab)
    assert np.array_equal(r["rgb"], rgb_to_u8(rgb)) and r["rgb"][0].tolist() == [0, 0, 255]
    assert np.array_equal(rgb_to_u8(np.array([0.5, 0.0, 1.0], np.float32)), [127, 0, 255])
    write_ply(p, V, F)
    r = read_ply(p)
    assert np.array_equal(r["verts"], V) and np.array_equal(r["faces"], F) and "rgb" not in r and "label" not in r

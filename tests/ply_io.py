"""Reader for the binary little-endian PLY files instance_nerf_b200.mesh.write_ply writes (tests only): parses the header
and the body with numpy."""
import numpy as np

_TYPES = {"float": "<f4", "uchar": "u1", "int": "<i4"}


def read_ply(path):
    """-> {"verts" [V, 3] f32, "faces" [F, 3] i32, "rgb" [V, 3] u8 (if present), "label" [V] i32 (if present)}"""
    with open(path, "rb") as f:
        data = f.read()
    end = data.index(b"end_header\n") + len(b"end_header\n")
    lines = data[:end].decode("ascii").splitlines()
    assert lines[0] == "ply" and lines[1] == "format binary_little_endian 1.0"
    elements, cur = [], None
    for ln in lines[2:-1]:
        w = ln.split()
        if w[0] == "element":
            cur = (w[1], int(w[2]), [])
            elements.append(cur)
        elif w[0] == "property" and w[1] == "list":
            assert w[2:] == ["uchar", "int", "vertex_indices"]
            cur[2].extend([("n", "u1"), ("v", "<i4", (3,))])
        elif w[0] == "property":
            cur[2].append((w[2], _TYPES[w[1]]))
    (vn, nv, vfields), (fn, nf, ffields) = elements
    assert vn == "vertex" and fn == "face"
    vrec = np.frombuffer(data, dtype=vfields, count=nv, offset=end)
    off = end + vrec.nbytes
    frec = np.frombuffer(data, dtype=ffields, count=nf, offset=off)
    assert off + frec.nbytes == len(data) and (frec["n"] == 3).all()
    out = {"verts": np.stack([vrec["x"], vrec["y"], vrec["z"]], 1), "faces": np.ascontiguousarray(frec["v"])}
    names = vrec.dtype.names
    if "red" in names:
        out["rgb"] = np.stack([vrec["red"], vrec["green"], vrec["blue"]], 1)
    if "label" in names:
        out["label"] = np.ascontiguousarray(vrec["label"])
    return out

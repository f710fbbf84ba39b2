"""Shared test fixtures: small synthetic scenes, rays, the canonical form of the reference's sample stream, and the
recorded outputs the GPU parity tests compare with."""
import functools
import hashlib
import os
import zlib

import numpy as np
import torch

from instance_nerf_b200 import synthetic
from oracle import host_oracle


@functools.lru_cache(maxsize=4)
def scene_arrays(K=16, bound=8.0, seed=0):
    sc = synthetic.RoomScene(K, bound, seed)
    cascade = 1 + int(np.ceil(np.log2(bound)))
    grid = sc.density_grid(cascade)
    bits = synthetic.packbits_np(grid, min(float(grid.mean()), 10.0))
    return sc, cascade, grid, bits


def make_rays(sc, H, W, n_poses=1, seed=1, pose_index=0):
    poses = synthetic.camera_poses(sc, max(n_poses, pose_index + 1), seed)[pose_index:pose_index + n_poses]
    r = host_oracle.get_rays(torch.from_numpy(poses), synthetic.intrinsics(H, W), H, W)
    return r["rays_o"].reshape(-1, 3).contiguous(), r["rays_d"].reshape(-1, 3).contiguous()


def adversarial_rays(bound):
    """Axis-parallel directions (rd = inf), rays grazing cell faces, rays starting outside / missing the box."""
    o, d = [], []
    for ax in range(3):
        for sgn in (1.0, -1.0):
            dd = [0.0, 0.0, 0.0]; dd[ax] = sgn
            o.append([0.1, -0.2, 0.3]); d.append(dd)
            oo = [0.0, 0.0, 0.0]; oo[(ax + 1) % 3] = 1.0 / 64  # exactly on a cell face of cascade 0
            o.append(oo); d.append(dd)
    o.append([20.0, 20.0, 20.0]); d.append([0.0, 1.0, 0.0])      # misses the aabb
    o.append([-20.0, 0.3, 0.1]); d.append([1.0, 0.0, 0.0])       # starts outside, hits
    o.append([0.0, 0.0, 0.0]); d.append([0.57735027, 0.57735027, 0.57735027])
    o.append([bound, bound, bound]); d.append([-0.57735027, -0.57735027, -0.57735027])
    return torch.tensor(o, dtype=torch.float32), torch.tensor(d, dtype=torch.float32)


def canonicalize(rays, xyzs, dirs, deltas, M=None):
    """SURVEY.md section 8a row 3: sort `rays` by ray id, offsets := exclusive prefix sum of counts, samples
    re-packed in that order.  Inputs may be torch (any device) or numpy; returns numpy."""
    rays, xyzs, dirs, deltas = (t.detach().cpu().numpy() if isinstance(t, torch.Tensor) else np.asarray(t) for t in (rays, xyzs, dirs, deltas))
    order = np.argsort(rays[:, 0], kind="stable")
    rays = rays[order]
    counts = rays[:, 2].astype(np.int64)
    old_off = rays[:, 1].astype(np.int64)
    new_off = np.concatenate([[0], np.cumsum(counts)[:-1]])
    total = int(counts.sum())
    cx = np.zeros((total, 3), np.float32); cd = np.zeros((total, 3), np.float32); cl = np.zeros((total, 2), np.float32)
    limit = xyzs.shape[0] if M is None else M
    for o, n, c in zip(old_off, new_off, counts):
        if c and o + c <= limit:
            cx[n:n + c] = xyzs[o:o + c]; cd[n:n + c] = dirs[o:o + c]; cl[n:n + c] = deltas[o:o + c]
    out_rays = np.stack([rays[:, 0], new_off, counts], -1).astype(np.int32)
    return out_rays, cx, cd, cl


def bits_equal(a, b):
    a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
    b = b.detach().cpu().numpy() if isinstance(b, torch.Tensor) else np.asarray(b)
    if a.shape != b.shape:
        return False
    if a.dtype.kind == "f":
        return np.array_equal(a.view(np.uint32 if a.itemsize == 4 else np.uint16), b.view(np.uint32 if b.itemsize == 4 else np.uint16))
    return np.array_equal(a, b)


GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _np(t):
    return t.detach().cpu().numpy() if isinstance(t, torch.Tensor) else np.asarray(t)


class Recorded:
    """What one GPU parity test compares the product with, kept in tests/golden/recorded_<test module>.npz.

    These tests used to run the reference's own CUDA kernels (oracle/_ref, compiled from the reference's sources, which are
    not part of this repository) next to the product's on the same inputs.  The reference side is stored instead.  It was
    recorded from this project's kernels at a commit where every one of these tests passed against the reference kernels,
    so it is the reference's output bit for bit where a test asks for that, and within the test's tolerance elsewhere.

    exact(name, t)   t must equal the recorded output bit for bit (stored as dtype, shape and SHA-256 of the bytes)
    close(name, t)   t must match the recorded output within (rtol, atol) on a fixed sample of its elements: all of them
                     for a small output, else `sample` seeded positions plus `sample` positions where it was non-zero
    value(name, v)   the recorded value of a small array or scalar

    With INERF_RECORD_GOLDEN=DIR set, the same calls store what they are given and the files are written to DIR when the
    session ends."""

    def __init__(self, store, prefix, record):
        self.store, self.prefix, self.record = store, prefix, record

    def _key(self, name):
        return f"{self.prefix}::{name}"

    def _get(self, name):
        k = self._key(name)
        if k not in self.store:
            raise KeyError(f"{k} is not recorded under tests/golden (see helpers.Recorded)")
        return self.store[k]

    def exact(self, name, t):
        a = np.ascontiguousarray(_np(t))
        h = f"{a.dtype.str}{list(a.shape)}:{hashlib.sha256(a.tobytes()).hexdigest()}"
        if self.record:
            self.store[self._key(name)] = np.array(h)
        else:
            want = str(self._get(name))
            assert h == want, f"{name}: differs from the recorded output ({h} vs {want})"

    def close(self, name, t, rtol, atol, equal_nan=False, sample=128):
        flat = _np(t).reshape(-1)
        if self.record:
            if flat.size <= 2 * sample:
                idx = np.arange(flat.size)
            else:
                rng = np.random.RandomState(zlib.crc32(self._key(name).encode()))
                nz = np.flatnonzero(flat)
                idx = np.unique(np.concatenate([rng.choice(flat.size, sample, replace=False),
                                                rng.choice(nz, min(sample, nz.size), replace=False)]))
            self.store[self._key(name + "#shape")] = np.array(_np(t).shape, np.int64)
            self.store[self._key(name + "#idx")] = idx.astype(np.int32 if flat.size < 2 ** 31 else np.int64)
            self.store[self._key(name + "#val")] = flat[idx]
            return
        assert tuple(_np(t).shape) == tuple(self._get(name + "#shape")), name
        idx = self._get(name + "#idx")
        torch.testing.assert_close(torch.from_numpy(np.ascontiguousarray(flat[idx])), torch.from_numpy(self._get(name + "#val")),
                                   rtol=rtol, atol=atol, equal_nan=equal_nan, msg=lambda m: f"{name}: {m}")

    def value(self, name, v):
        if self.record:
            self.store[self._key(name)] = np.asarray(v)
            return v
        return self._get(name)


def record_metric(name, **kv):
    """Append a measured figure of a GPU test to gpurun_out/test_metrics.jsonl (brought back by gpurun; best effort)."""
    import json
    import os
    try:
        root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
        os.makedirs(os.path.join(root, "gpurun_out"), exist_ok=True)
        with open(os.path.join(root, "gpurun_out", "test_metrics.jsonl"), "a") as f:
            f.write(json.dumps({"test": name, **kv}) + "\n")
    except OSError:
        pass
